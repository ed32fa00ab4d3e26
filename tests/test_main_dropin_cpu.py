"""The unchanged reference main.py (main.py:1-121) imports and constructs everything from OUR packages
(facade models, agent classes, Grid_World) and hands them to OUR train_RPBCAC.  No GPU is needed up to that call, so
the training function is intercepted here; the GPU part of the contract is covered by tests/test_api_gpu.py.
The driver comes out of tests/golden/ref_main_py.npz (byte-identical, SHA-256 checked)."""
import os
import sys

import numpy as np
import pandas as pd

from golden_util import write_reference_main

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_main_runs_unchanged_on_our_packages(tmp_path, monkeypatch):
    ref_main = write_reference_main(tmp_path)
    dropin = os.path.join(ROOT, "resilient-consensus-based-marl_b200")
    sys.path.insert(0, dropin)
    import run_main
    import training.train_agents as training
    seen = {}

    def fake_train(env, agents, args, exp_buffer=None):
        seen.update(env=env, agents=agents, args=args)
        w = np.empty(len(agents), dtype=object)
        for i, a in enumerate(agents):
            w[i] = a.get_parameters()
        return w, pd.DataFrame([{"True_team_returns": 0.0, "True_adv_returns": 0.0, "Estimated_team_returns": 0.0}])
    monkeypatch.setattr(training, "train_RPBCAC", fake_train)
    monkeypatch.chdir(tmp_path)                      # main.py writes its artefacts to the cwd (main.py:119-121)
    run_main.main(["run_main.py", ref_main, "--H=1", "--slow_lr=0.002", "--random_seed=100", "--n_episodes=50"])
    from agents.resilient_CAC_agents import RPBCAC_agent
    from environments.grid_world import Grid_World
    assert type(seen["env"]) is Grid_World and seen["env"].__class__.__module__ == "environments.grid_world"
    assert os.path.realpath(sys.modules["agents.resilient_CAC_agents"].__file__).startswith(os.path.realpath(dropin))
    assert len(seen["agents"]) == 5 and all(isinstance(a, RPBCAC_agent) for a in seen["agents"])
    assert seen["agents"][0].H == 1 and seen["agents"][0].fast_lr == 0.01 and seen["args"]["slow_lr"] == 0.002
    assert [x.shape for x in seen["agents"][0].get_parameters()[2]] == [(15, 20), (20,), (20, 20), (20,), (20, 1), (1,)]
    # same NumPy draws as the reference before training starts (main.py:46-49)
    np.random.seed(100)
    assert np.array_equal(np.load(tmp_path / "desired_state.npy"), np.random.randint(0, 5, size=(5, 2)))
    back = np.load(tmp_path / "pretrained_weights.npy", allow_pickle=True)
    assert back.shape == (5,) and os.path.exists(tmp_path / "sim_data.pkl")
