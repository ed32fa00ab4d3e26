"""Helpers shared by the tests: load golden fixtures (tests/golden/*.npz)."""
import hashlib
import os
import zlib

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def agent_weights(z, prefix, n_agents=5):
    """-> list over agents of list over nets (actor, critic, TR[, critic_local]) of 6 arrays."""
    out = []
    for i in range(n_agents):
        nets = []
        n = 0
        while f"{prefix}/agent{i}/n{n}_k0" in z.files:
            nets.append([z[f"{prefix}/agent{i}/n{n}_k{k}"] for k in range(6)])
            n += 1
        out.append(nets)
    return out


def pretrained(tag="malicious_H1_s100"):
    z = load("kat_est_returns.npz")
    return agent_weights(z, tag), z[f"{tag}/desired"], [str(x) for x in z[f"{tag}/labels"]]


def write_reference_main(directory):
    """The reference driver main.py out of ref_main_py.npz, checked against its stored SHA-256, as directory/main.py."""
    z = load("ref_main_py.npz")
    raw = zlib.decompress(z["blob"].tobytes())
    assert hashlib.sha256(raw).hexdigest() == str(z["sha256"]) and len(raw) == int(z["n_bytes"])
    script = os.path.join(directory, "main.py")
    with open(script, "wb") as f:
        f.write(raw)
    return script
