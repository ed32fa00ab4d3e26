"""The UNCHANGED reference driver (main.py of mfigura/Resilient-consensus-based-MARL, byte-identical: SHA-256 checked) runs
end to end on the drop-in packages through REAL training on the GPU: argparse -> model / agent / env construction
(main.py:59-116) -> training.train_RPBCAC (main.py:117) -> the three artefacts (main.py:119-121).  The driver comes out of
tests/golden/ref_main_py.npz (a compressed blob written by oracle/make_golden.py; the GPU box has no reference checkout)."""
import os
import sys

import numpy as np
import pandas as pd
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from golden_util import write_reference_main            # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("n_envs,flags", [(1, ["--H=1", "--slow_lr=0.002", "--random_seed=100"]),
                                          (64, ["--H=0", "--random_seed=300", "--n_agents=5"])])
def test_reference_main_trains_end_to_end_unchanged(n_envs, flags, tmp_path, monkeypatch, capsys):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    script = write_reference_main(tmp_path)
    dropin = os.path.join(ROOT, "resilient-consensus-based-marl_b200")
    sys.path.insert(0, dropin)
    import run_main
    monkeypatch.chdir(tmp_path)                                   # the driver writes its artefacts to the cwd
    monkeypatch.setenv("RCMARL_N_ENVS", str(n_envs))
    run_main.main(["run_main.py", str(script), "--n_episodes=100"] + flags)
    out = capsys.readouterr().out
    assert out.count("| Episode:") == 100                        # the reference's per-episode log line (train_agents.py:174)
    sim = pd.read_pickle(tmp_path / "sim_data.pkl")               # main.py:119
    assert list(sim.columns) == ["True_team_returns", "True_adv_returns", "Estimated_team_returns"] and len(sim) == 100
    assert np.isfinite(sim.to_numpy()).all() and (sim["True_team_returns"] < 0).all()
    w = np.load(tmp_path / "pretrained_weights.npy", allow_pickle=True)          # main.py:120
    assert w.shape == (5,) and all(len(w[i]) == 3 for i in range(5))
    for i in range(5):
        assert [a.shape for a in w[i][0]] == [(10, 20), (20,), (20, 20), (20,), (20, 5), (5,)]
        assert [a.shape for a in w[i][1]] == [(10, 20), (20,), (20, 20), (20,), (20, 1), (1,)]
        assert [a.shape for a in w[i][2]] == [(15, 20), (20,), (20, 20), (20,), (20, 1), (1,)]
        assert all(np.isfinite(a).all() for net in w[i] for a in net)
    seed = int([f for f in flags if f.startswith("--random_seed")][0].split("=")[1])
    np.random.seed(seed)
    assert np.array_equal(np.load(tmp_path / "desired_state.npy"), np.random.randint(0, 5, size=(5, 2)))   # main.py:48,121
    # two update rounds happened (episodes 49 and 99): the trained critics differ from each other and moved
    assert not np.allclose(w[0][1][0], w[1][1][0])
