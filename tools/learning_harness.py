"""Learning-curve reproduction harness (SURVEY 8f.2, README.md:31-45 of the reference): every published run directory
(8 scenarios x H in {0, 1} x seeds {100, 200, 300}; 45 exist) is re-run from ITS OWN start weights and task
(tests/golden/ref_learning/<scenario>.npz, extracted by oracle/make_golden.py -- no reference checkout is needed), and the mean
of the last 500 episodes is printed next to the mean of the last 500 episodes of the reference's sim_data2.pkl.

    python tools/learning_harness.py [n_blocks=40] [n_envs=256] [filter]      -> gpurun_out/learning_harness.{json,md}

The comparison is qualitative by construction (the published runs trained one environment for 8 000 episodes with an older
code version, SURVEY 6): the reproduced claims are
  (1) under attack (faulty / greedy / malicious, local or team-average rewards) H = 1 keeps the cooperative team's return
      near the attack-free level while H = 0 does not, and
  (2) with H = 0 the malicious agent drives the cooperative critics' estimate of the team return far above the truth.
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "resilient-consensus-based-marl_b200"))
import bench                                   # noqa: E402
from rcmarl.trainer import Trainer             # noqa: E402

n_blocks = int(sys.argv[1]) if len(sys.argv) > 1 else 40
n_envs = int(sys.argv[2]) if len(sys.argv) > 2 else 256
only = sys.argv[3] if len(sys.argv) > 3 else ""
golden = os.path.join(ROOT, "tests", "golden", "ref_learning")
runs = []                                       # (run tag, the scenario's fixture holding it)
for name in sorted(os.listdir(golden)):
    z = np.load(os.path.join(golden, name))
    runs += [(str(r), z) for r in z["runs"] if only in str(r)]
tail = 10                                       # 10 blocks x 50 episodes = the last 500 episodes
rows = []
for tag, z in runs:
    scen, Hs, ss = tag.split("/")
    H, seed = int(Hs[1:]), int(ss[1:])
    labels = [str(x) for x in z[f"{tag}/labels"]]
    w = []
    for i in range(len(labels)):
        nets_i, n = [], 0
        while f"{tag}/agent{i}/n{n}_k0" in z.files:
            nets_i.append([z[f"{tag}/agent{i}/n{n}_k{k}"] for k in range(6)])
            n += 1
        w.append(nets_i)
    tr = Trainer(labels=labels, in_nodes=bench.IN_NODES5, weights=w, desired=z[f"{tag}/desired"], n_envs=n_envs, H=H, seed=seed,
                 common_reward=bool(z[f"{tag}/common_reward"]), **bench.HYPER)
    coop = [i for i, l in enumerate(labels) if l == "Cooperative"]
    adv = [i for i, l in enumerate(labels) if l != "Cooperative"]
    team, est, advr = [], [], []
    for b in range(n_blocks):
        e, r = tr.rollout_block()
        tr.update_round()
        team.append(float(r[:, coop].mean())); est.append(float(e[:, coop].mean()))
        advr.append(float(r[:, adv].mean()) if adv else 0.0)
    row = dict(run=tag, scenario=scen, H=H, seed=seed, ours_team=float(np.mean(team[-tail:])), ours_est=float(np.mean(est[-tail:])),
               ours_adv=float(np.mean(advr[-tail:])), first_team=team[0], ref_team=float(z[f"{tag}/ref_team"]),
               ref_est=float(z[f"{tag}/ref_est"]), ref_adv=float(z[f"{tag}/ref_adv"]), team_curve=team, est_curve=est)
    rows.append(row)
    print(f"{tag:28s} ours: team {row['ours_team']:6.2f} est {row['ours_est']:6.2f} adv {row['ours_adv']:6.2f} | "
          f"reference: team {row['ref_team']:6.2f} est {row['ref_est']:6.2f} adv {row['ref_adv']:6.2f}", flush=True)

# ---- per (scenario, H): means over seeds, ours vs reference, and the two qualitative claims
summary = {}
for scen in sorted({r["scenario"] for r in rows}):
    for H in (0, 1):
        sel = [r for r in rows if r["scenario"] == scen and r["H"] == H]
        if sel:
            summary[f"{scen}/H={H}"] = {k: float(np.mean([r[k] for r in sel])) for k in
                                        ("ours_team", "ours_est", "ours_adv", "ref_team", "ref_est", "ref_adv")} | {"seeds": len(sel)}
checks = []
for scen in ("faulty", "greedy", "malicious", "faulty_global", "greedy_global", "malicious_global"):
    a, b = summary.get(f"{scen}/H=0"), summary.get(f"{scen}/H=1")
    if a and b:
        checks.append(dict(claim=f"{scen}: H=1 team return above H=0", ours=b["ours_team"] - a["ours_team"],
                           reference=b["ref_team"] - a["ref_team"], holds=bool(b["ours_team"] > a["ours_team"])))
for scen in ("malicious", "malicious_global"):
    a = summary.get(f"{scen}/H=0")
    if a:
        checks.append(dict(claim=f"{scen} H=0: critic estimate poisoned above the true return", ours=a["ours_est"] - a["ours_team"],
                           reference=a["ref_est"] - a["ref_team"], holds=bool(a["ours_est"] - a["ours_team"] > 2.0)))
os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
json.dump(dict(n_blocks=n_blocks, n_envs=n_envs, runs=rows, summary=summary, checks=checks),
          open(os.path.join(ROOT, "gpurun_out", "learning_harness.json"), "w"))
with open(os.path.join(ROOT, "gpurun_out", "learning_harness.md"), "w") as f:
    f.write(f"| scenario / H | seeds | ours team | ref team | ours estimate | ref estimate | ours adversary | ref adversary |\n|---|---|---|---|---|---|---|---|\n")
    for k, v in summary.items():
        f.write(f"| {k} | {v['seeds']} | {v['ours_team']:.2f} | {v['ref_team']:.2f} | {v['ours_est']:.2f} | {v['ref_est']:.2f} | "
                f"{v['ours_adv']:.2f} | {v['ref_adv']:.2f} |\n")
    f.write("\n| claim | ours | reference | holds |\n|---|---|---|---|\n")
    for c in checks:
        f.write(f"| {c['claim']} | {c['ours']:.2f} | {c['reference']:.2f} | {c['holds']} |\n")
print(open(os.path.join(ROOT, "gpurun_out", "learning_harness.md")).read())
