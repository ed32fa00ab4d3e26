"""Generate tests/golden/*.npz -- TEST INFRASTRUCTURE, run only in the authoring
container (needs /root/reference, which does not exist on the GPU box).

    python oracle/make_golden.py

1. kat_est_returns.npz     known-answer vectors logged by the *real* TF run of
                           the reference (simulation_results/raw_data/**/out.txt,
                           SURVEY.md Appendix B) + the weights they belong to.
2. ref_methods.npz         every RPBCAC_agent / Malicious_CAC_agent method of the
                           reference sources, executed VERBATIM from
                           /root/reference on oracle/tf_facade, on seeded inputs.
3. ref_train_run.npz       reference training/train_agents.py:train_RPBCAC run
                           verbatim (2 update rounds, 4 coop + 1 malicious, H=1):
                           replay buffer, injected fit permutations, final weights.
4. ref_env.npz             reference environments/grid_world.py transitions.
5. ref_adversaries.npz     every Greedy_CAC_agent / Faulty_CAC_agent method
                           (agents/adversarial_CAC_agents.py:5-72,184-275) executed
                           verbatim on seeded inputs with injected fit permutations,
                           plus train_RPBCAC verbatim for 3 cooperative + 1 greedy +
                           1 faulty agent with common_reward=True (2 update rounds).
7. ref_main_py.npz         the reference driver main.py as a compressed blob (executed unchanged by tests/test_main_*.py).
6. ref_learning/*.npz      start weights / task / last-500-episode means of sim_data2.pkl
                           for the 45 published run directories (tools/learning_harness.py).
"""
import os
import re
import sys
import io
import contextlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("RCMARL_REFERENCE", "/root/reference")
OUT = os.path.join(ROOT, "tests", "golden")

sys.path.insert(0, os.path.join(HERE, "tf_facade"))
sys.path.insert(1, REF)

import tensorflow as tf                                   # noqa: E402  (the facade)
from tensorflow import keras                              # noqa: E402
from environments.grid_world import Grid_World            # noqa: E402  (reference, verbatim)
from agents.resilient_CAC_agents import RPBCAC_agent      # noqa: E402
from agents.adversarial_CAC_agents import Malicious_CAC_agent, Greedy_CAC_agent, Faulty_CAC_agent   # noqa: E402
import training.train_agents as ref_training              # noqa: E402

RAW = os.path.join(REF, "simulation_results", "raw_data")


def flat_weights(w_agent):
    """object array entry -> dict of named float32 arrays."""
    out = {}
    for n, net in enumerate(w_agent):
        for k, arr in enumerate(net):
            out[f"n{n}_k{k}"] = np.asarray(arr, np.float32)
    return out


def parse_est_returns(path, n):
    pat = re.compile(r"\| Episode: (\d+) \| Est\. returns: \[([^\]]*)\]")
    rows = []
    with open(path) as f:
        for line in f:
            m = pat.match(line)
            if m:
                rows.append([float(x) for x in m.group(2).split(",")])
                if len(rows) == n:
                    break
    return rows


def make_kat():
    runs = [("malicious", 1, 100, "pretrained_weights.npy"),
            ("coop", 0, 200, "pretrained_weights.npy"),
            ("greedy", 1, 300, "pretrained_weights.npy"),
            ("faulty_global", 1, 100, "pretrained_weights1.npy")]
    out = {}
    for scen, H, seed, wfile in runs:
        d = os.path.join(RAW, scen, f"H={H}", f"seed={seed}")
        w = np.load(os.path.join(d, wfile), allow_pickle=True)
        tag = f"{scen}_H{H}_s{seed}"
        with open(os.path.join(d, "out.txt")) as f:
            head = f.read(4000)
        labels = re.search(r"'agent_label': \[([^\]]*)\]", head).group(1).replace("'", "").replace(" ", "").split(",")
        out[f"{tag}/labels"] = np.array(labels)
        out[f"{tag}/seed"] = np.int64(seed)
        # the desired state is printed right after the args dict (main.py:106)
        dtxt = re.search(r"\}\s*(\[\[.*?\]\])", head, re.S).group(1)
        desired = np.array([[int(v) for v in row.split()] for row in re.findall(r"\[([\d\s]+)\]", dtxt)], np.int64)
        dfile = os.path.join(d, "desired_state.npy")
        if os.path.exists(dfile):
            assert np.array_equal(desired, np.load(dfile, allow_pickle=True))
        out[f"{tag}/desired"] = desired
        est = parse_est_returns(os.path.join(d, "out.txt"), 50)
        out[f"{tag}/est_returns"] = np.array(est, np.float64)
        for i in range(len(w)):
            for k, v in flat_weights(w[i]).items():
                out[f"{tag}/agent{i}/{k}"] = v
    np.savez_compressed(os.path.join(OUT, "kat_est_returns.npz"), **out)
    print("kat:", len(out), "arrays")


def build_models(w_agent, n_agents=5, n_actions=5):
    def seq(d_feat, n_out, act):
        return keras.Sequential([keras.Input(shape=(n_agents, d_feat)), keras.layers.Flatten(),
                                 keras.layers.Dense(20, activation=keras.layers.LeakyReLU(alpha=0.1)),
                                 keras.layers.Dense(20, activation=keras.layers.LeakyReLU(alpha=0.1)),
                                 keras.layers.Dense(n_out, activation=act)])
    actor, critic, tr = seq(2, n_actions, 'softmax'), seq(2, 1, None), seq(3, 1, None)
    actor.set_weights(w_agent[0])
    critic.set_weights(w_agent[1])
    tr.set_weights(w_agent[2])
    return actor, critic, tr


def load_w():
    d = os.path.join(RAW, "malicious", "H=1", "seed=100")
    return np.load(os.path.join(d, "pretrained_weights.npy"), allow_pickle=True), \
        np.load(os.path.join(d, "desired_state.npy"), allow_pickle=True)


def synth_batch(rs, B, n_agents=5):
    pos = rs.randint(0, 5, size=(B, n_agents, 2))
    npos = np.clip(pos + rs.randint(-1, 2, size=pos.shape), 0, 4)
    s = ((pos - 2.0) / np.std(np.arange(5))).astype(np.float32)
    ns = ((npos - 2.0) / np.std(np.arange(5))).astype(np.float32)
    a = rs.randint(0, 5, size=(B, n_agents, 1)).astype(np.float32)
    r = (-rs.randint(0, 9, size=(B, n_agents, 1)) / 5.0).astype(np.float32)
    return s, ns, a, r


def make_methods():
    w, _ = load_w()
    rs = np.random.RandomState(7)
    B = 96
    s, ns, a, r = synth_batch(rs, B)
    sa = np.concatenate([s, a], -1)
    out = dict(s=s, ns=ns, a=a, r=r)
    S, NS, SA = (tf.convert_to_tensor(x, tf.float32) for x in (s, ns, sa))
    R = tf.convert_to_tensor(r, tf.float32)
    for H in (0, 1):
        actor, critic, tr = build_models(w[0])
        ag = RPBCAC_agent(actor, critic, tr, slow_lr=0.002, fast_lr=0.01, gamma=0.9, H=H)
        cw, closs = ag.critic_update_local(S, NS, R[:, 0])
        tw, tloss = ag.TR_update_local(SA, R[:, 0])
        for k in range(6):
            out[f"H{H}/critic_local_k{k}"] = cw[k]
            out[f"H{H}/tr_local_k{k}"] = tw[k]
        out[f"H{H}/critic_local_loss"] = np.float32(closs)
        out[f"H{H}/tr_local_loss"] = np.float32(tloss)
        # unchanged-after-local check
        out[f"H{H}/critic_after_local_same"] = np.array(
            all(np.array_equal(x, y) for x, y in zip(critic.get_weights(), w[0][1])))
        # messages: own locally-updated + three other agents' pretrained nets
        cmsgs = [cw] + [list(w[j][1]) for j in (1, 2, 4)]
        tmsgs = [tw] + [list(w[j][2]) for j in (1, 2, 4)]
        ag.resilient_consensus_critic_hidden(cmsgs)
        ag.resilient_consensus_TR_hidden(tmsgs)
        for k, arr in enumerate(critic.get_weights()):
            out[f"H{H}/critic_after_hidden_k{k}"] = arr
        for k, arr in enumerate(tr.get_weights()):
            out[f"H{H}/tr_after_hidden_k{k}"] = arr
        cagg = ag.resilient_consensus_critic(S, cmsgs)
        tagg = ag.resilient_consensus_TR(SA, tmsgs)
        out[f"H{H}/critic_agg"] = np.asarray(cagg)
        out[f"H{H}/tr_agg"] = np.asarray(tagg)
        ag.critic_update_team(S, cagg)
        ag.TR_update_team(SA, tagg)
        for k, arr in enumerate(critic.get_weights()):
            out[f"H{H}/critic_after_team_k{k}"] = arr
        for k, arr in enumerate(tr.get_weights()):
            out[f"H{H}/tr_after_team_k{k}"] = arr
        for step in range(3):                      # Adam state persists across calls
            al = ag.actor_update(S, NS, SA, tf.convert_to_tensor(a, tf.float32)[:, 0])
            out[f"H{H}/actor_loss_{step}"] = np.float32(al)
            for k, arr in enumerate(actor.get_weights()):
                out[f"H{H}/actor_after_{step}_k{k}"] = arr
        probs = actor.predict(s[:8])
        out[f"H{H}/probs"] = probs
    # aggregation on its own, incl. ties and n < 2H+2
    ag0 = RPBCAC_agent(*build_models(w[0]), slow_lr=0.002, fast_lr=0.01, gamma=0.9, H=0)
    for n, H in ((4, 0), (4, 1), (6, 2), (9, 4), (3, 1)):
        v = rs.randn(n, 37).astype(np.float32)
        v[:, ::5] = np.round(v[:, ::5])
        ag0.H = H
        out[f"agg/n{n}_H{H}_in"] = v
        out[f"agg/n{n}_H{H}_out"] = np.asarray(ag0._resilient_aggregation(tf.convert_to_tensor(v)))
    # Malicious methods with injected permutations
    perm_rs = np.random.RandomState(11)
    used = []

    def hook(Bn):
        p = perm_rs.permutation(Bn)
        used.append(p)
        return p
    tf.perm_hook = hook
    actor, critic, tr = build_models(w[4])
    mal = Malicious_CAC_agent(actor, critic, tr, slow_lr=0.002, fast_lr=0.01, gamma=0.9)
    mal.critic_local_weights = w[4][3]
    mal.critic_update_local(S, NS, R[:, 4])
    x, xl = mal.TR_update_compromised(SA, -R[:, 0])
    y, yl = mal.critic_update_compromised(S, NS, -R[:, 0])
    big = [np.concatenate([t] * 3, 0) for t in (s, ns, r, a)]          # 288 rows -> 2 actor mini-batches
    al = mal.actor_update(tf.convert_to_tensor(big[0]), tf.convert_to_tensor(big[1]),
                          tf.convert_to_tensor(big[2])[:, 4], tf.convert_to_tensor(big[3])[:, 4])
    tf.perm_hook = None
    for k in range(6):
        out[f"mal/critic_local_k{k}"] = mal.critic_local_weights[k]
        out[f"mal/tr_k{k}"] = x[k]
        out[f"mal/critic_k{k}"] = y[k]
        out[f"mal/actor_k{k}"] = actor.get_weights()[k]
    out["mal/tr_loss"], out["mal/critic_loss"], out["mal/actor_loss"] = np.float32(xl), np.float32(yl), np.float32(al)
    out["mal/perms_96"] = np.stack(used[:30])
    out["mal/perm_288"] = used[30]
    np.savez_compressed(os.path.join(OUT, "ref_methods.npz"), **out)
    print("methods:", len(out), "arrays")


def make_train_run():
    w, desired = load_w()
    labels = ['Cooperative'] * 4 + ['Malicious']
    in_nodes = [[0, 1, 2, 3], [1, 2, 3, 4], [2, 3, 4, 0], [3, 4, 0, 1], [4, 0, 1, 2]]
    args = dict(n_agents=5, agent_label=labels, in_nodes=in_nodes, n_actions=5, n_states=2,
                n_episodes=50, max_ep_len=10, n_ep_fixed=25, n_epochs=2, slow_lr=0.002, fast_lr=0.01,
                batch_size=200, buffer_size=100000, gamma=0.9, H=1, common_reward=False)
    np.random.seed(5)
    tf.random.set_seed(5)
    agents = []
    for i in range(5):
        actor, critic, tr = build_models(w[i])
        if labels[i] == 'Malicious':
            ag = Malicious_CAC_agent(actor, critic, tr, slow_lr=0.002, fast_lr=0.01, gamma=0.9)
            ag.critic_local_weights = w[i][3]
        else:
            ag = RPBCAC_agent(actor, critic, tr, slow_lr=0.002, fast_lr=0.01, gamma=0.9, H=1)
        agents.append(ag)
    env = Grid_World(nrow=5, ncol=5, n_agents=5, desired_state=desired,
                     initial_state=np.zeros((5, 2), int), randomize_state=True, scaling=True)
    perm_rs = np.random.RandomState(21)
    used = []

    def hook(Bn):
        p = perm_rs.permutation(Bn)
        used.append(p)
        return p
    tf.perm_hook = hook
    buf = [[], [], [], []]
    buf_probe = buf
    with contextlib.redirect_stdout(io.StringIO()):
        weights, sim = ref_training.train_RPBCAC(env, agents, args, exp_buffer=buf_probe)
    tf.perm_hook = None
    out = dict(desired=np.asarray(desired, np.int64),
               s=np.asarray(buf[0], np.float32), ns=np.asarray(buf[1], np.float32),
               a=np.asarray(buf[2], np.float32), r=np.asarray(buf[3], np.float32),
               est=sim["Estimated_team_returns"].to_numpy(), ret=sim["True_team_returns"].to_numpy(),
               ret_adv=sim["True_adv_returns"].to_numpy())
    out["n_perms"] = np.int64(len(used))
    for j, p in enumerate(used):
        out[f"perm{j}"] = p
    for i in range(5):
        for n, net in enumerate(weights[i]):
            for k, arr in enumerate(net):
                out[f"final/agent{i}/n{n}_k{k}"] = np.asarray(arr, np.float32)
    np.savez_compressed(os.path.join(OUT, "ref_train_run.npz"), **out)
    print("train run: rows", out["s"].shape, "perms", len(used))


def make_env():
    rs = np.random.RandomState(3)
    out = {}
    for tag, nrow, na in (("5x5", 5, 5), ("10x10", 10, 16), ("3x3", 3, 3)):
        desired = rs.randint(0, nrow, size=(na, 2))
        env = Grid_World(nrow=nrow, ncol=nrow, n_agents=na, desired_state=desired,
                         initial_state=np.zeros((na, 2), int), randomize_state=True, scaling=True)
        env.state = desired.copy()                      # start on the goal: exercises the reward==0 branch
        S, A, R, SS = [env.state.copy()], [], [], []
        for t in range(60):
            act = rs.randint(0, 5, size=na).astype(float)
            if t < 3:
                act[:] = 0
            env.step(act)
            st, rw = env.get_data()
            A.append(act)
            R.append(rw.copy())
            SS.append(st.copy())
            S.append(env.state.copy())
        out[f"{tag}/desired"] = desired
        out[f"{tag}/state_int"] = np.array(S)
        out[f"{tag}/action"] = np.array(A)
        out[f"{tag}/reward_scaled"] = np.array(R)
        out[f"{tag}/state_scaled"] = np.array(SS)
    np.savez_compressed(os.path.join(OUT, "ref_env.npz"), **out)
    print("env:", len(out), "arrays")


def make_adversaries():
    """Greedy_CAC_agent / Faulty_CAC_agent (agents/adversarial_CAC_agents.py:184-275, :5-72) method vectors and a
    verbatim train_RPBCAC run with both of them and common_reward=True (the *_global scenarios, train_agents.py:106)."""
    w, desired = load_w()
    rs = np.random.RandomState(17)
    B = 96
    s, ns, a, r = synth_batch(rs, B)
    sa = np.concatenate([s, a], -1)
    out = dict(s=s, ns=ns, a=a, r=r)
    S, NS, SA = (tf.convert_to_tensor(x, tf.float32) for x in (s, ns, sa))
    R = tf.convert_to_tensor(r, tf.float32)
    perm_rs = np.random.RandomState(19)
    used = []

    def hook(Bn):
        p = perm_rs.permutation(Bn)
        used.append(p)
        return p
    tf.perm_hook = hook
    # ---- Greedy: critic / TR mini-batch fits on the local reward, actor fit(batch 200)
    actor, critic, tr = build_models(w[3])
    gr = Greedy_CAC_agent(actor, critic, tr, slow_lr=0.002, fast_lr=0.01, gamma=0.9)
    x, xl = gr.TR_update_local(SA, R[:, 3])
    y, yl = gr.critic_update_local(S, NS, R[:, 3])
    big = [np.concatenate([t] * 3, 0) for t in (s, ns, r, a)]          # 288 rows -> 2 actor mini-batches
    al = gr.actor_update(tf.convert_to_tensor(big[0]), tf.convert_to_tensor(big[1]),
                         tf.convert_to_tensor(big[2])[:, 3], tf.convert_to_tensor(big[3])[:, 3])
    for k in range(6):
        out[f"greedy/tr_k{k}"] = x[k]
        out[f"greedy/critic_k{k}"] = y[k]
        out[f"greedy/actor_k{k}"] = actor.get_weights()[k]
    out["greedy/tr_loss"], out["greedy/critic_loss"], out["greedy/actor_loss"] = np.float32(xl), np.float32(yl), np.float32(al)
    out["greedy/perms_96"] = np.stack(used[:20])
    out["greedy/perm_288"] = used[20]
    gp = gr.get_parameters()
    out["greedy/n_param_lists"] = np.int64(len(gp))
    del used[:]
    # ---- Faulty: only the actor learns; critic / TR are transmitted unchanged
    actor, critic, tr = build_models(w[4])
    fa = Faulty_CAC_agent(actor, critic, tr, slow_lr=0.002, gamma=0.9)
    al = fa.actor_update(tf.convert_to_tensor(big[0]), tf.convert_to_tensor(big[1]),
                         tf.convert_to_tensor(big[2])[:, 4], tf.convert_to_tensor(big[3])[:, 4])
    out["faulty/actor_loss"] = np.float32(al)
    out["faulty/perm_288"] = used[0]
    for k in range(6):
        out[f"faulty/actor_k{k}"] = actor.get_weights()[k]
        out[f"faulty/critic_k{k}"] = fa.get_critic_weights()[k]
        out[f"faulty/tr_k{k}"] = fa.get_TR_weights()[k]
    out["faulty/critic_unchanged"] = np.array(all(np.array_equal(p, q) for p, q in zip(fa.get_critic_weights(), w[4][1])))
    out["faulty/tr_unchanged"] = np.array(all(np.array_equal(p, q) for p, q in zip(fa.get_TR_weights(), w[4][2])))
    tf.perm_hook = None

    # ---- train_RPBCAC verbatim: 3 cooperative + greedy + faulty, team-average reward for everyone (common_reward)
    labels = ['Cooperative'] * 3 + ['Greedy', 'Faulty']
    in_nodes = [[0, 1, 2, 3], [1, 2, 3, 4], [2, 3, 4, 0], [3, 4, 0, 1], [4, 0, 1, 2]]
    args = dict(n_agents=5, agent_label=labels, in_nodes=in_nodes, n_actions=5, n_states=2,
                n_episodes=50, max_ep_len=10, n_ep_fixed=25, n_epochs=2, slow_lr=0.002, fast_lr=0.01,
                batch_size=200, buffer_size=100000, gamma=0.9, H=1, common_reward=True)
    np.random.seed(6)
    tf.random.set_seed(6)
    agents = []
    for i in range(5):
        actor, critic, tr = build_models(w[i])
        if labels[i] == 'Greedy':
            ag = Greedy_CAC_agent(actor, critic, tr, slow_lr=0.002, fast_lr=0.01, gamma=0.9)
        elif labels[i] == 'Faulty':
            ag = Faulty_CAC_agent(actor, critic, tr, slow_lr=0.002, gamma=0.9)
        else:
            ag = RPBCAC_agent(actor, critic, tr, slow_lr=0.002, fast_lr=0.01, gamma=0.9, H=1)
        agents.append(ag)
    env = Grid_World(nrow=5, ncol=5, n_agents=5, desired_state=desired,
                     initial_state=np.zeros((5, 2), int), randomize_state=True, scaling=True)
    perm_rs = np.random.RandomState(23)
    used = []
    tf.perm_hook = hook
    buf = [[], [], [], []]
    with contextlib.redirect_stdout(io.StringIO()):
        weights, sim = ref_training.train_RPBCAC(env, agents, args, exp_buffer=buf)
    tf.perm_hook = None
    out["run/desired"] = np.asarray(desired, np.int64)
    out["run/labels"] = np.array(labels)
    for name, arr in zip(("s", "ns", "a", "r"), buf):
        out[f"run/{name}"] = np.asarray(arr, np.float32)
    out["run/n_perms"] = np.int64(len(used))
    for j, p in enumerate(used):
        out[f"run/perm{j}"] = p
    for i in range(5):
        for n, net in enumerate(weights[i]):
            for k, arr in enumerate(net):
                out[f"run/final/agent{i}/n{n}_k{k}"] = np.asarray(arr, np.float32)
    np.savez_compressed(os.path.join(OUT, "ref_adversaries.npz"), **out)
    print("adversaries:", len(out), "arrays; train-run perms", len(used))


def make_learning_fixture():
    """Start weights, task and published outcome of every run directory under simulation_results/raw_data (8 scenarios
    x H in {0,1} x seeds {100,200,300}; 45 exist): the inputs of tools/learning_harness.py and the numbers it prints next
    to ours (README.md:31-45).  `ref_*` = mean over the last 500 episodes of sim_data2.pkl (run 2 of the published jobs).
    One file per scenario (ref_learning/<scenario>.npz) keeps each fixture well under 1 MB."""
    import pandas as pd
    os.makedirs(os.path.join(OUT, "ref_learning"), exist_ok=True)
    n_runs = 0
    for scen in sorted(os.listdir(RAW)):
        out, runs = {}, []
        for H in (0, 1):
            for seed in (100, 200, 300):
                d = os.path.join(RAW, scen, f"H={H}", f"seed={seed}")
                if not os.path.isdir(d):
                    continue
                wfile = "pretrained_weights1.npy" if os.path.exists(os.path.join(d, "pretrained_weights1.npy")) else "pretrained_weights.npy"
                w = np.load(os.path.join(d, wfile), allow_pickle=True)
                head = open(os.path.join(d, "out.txt")).read(4000)
                labels = re.search(r"'agent_label': \[([^\]]*)\]", head).group(1).replace("'", "").replace(" ", "").split(",")
                common = re.search(r"'common_reward': (\w+)", head).group(1) == "True"
                dtxt = re.search(r"\}\s*(\[\[.*?\]\])", head, re.S).group(1)
                desired = np.array([[int(v) for v in row.split()] for row in re.findall(r"\[([\d\s]+)\]", dtxt)], np.int64)
                df = pd.read_pickle(os.path.join(d, "sim_data2.pkl")).tail(500).mean()
                tag = f"{scen}/H{H}/s{seed}"
                runs.append(tag)
                out[f"{tag}/labels"] = np.array(labels)
                out[f"{tag}/common_reward"] = np.array(common)
                out[f"{tag}/desired"] = desired
                out[f"{tag}/ref_team"] = np.float64(df["True_team_returns"])
                out[f"{tag}/ref_adv"] = np.float64(df["True_adv_returns"])
                out[f"{tag}/ref_est"] = np.float64(df["Estimated_team_returns"])
                for i in range(len(w)):
                    for k, v in flat_weights(w[i]).items():
                        out[f"{tag}/agent{i}/{k}"] = v
        if runs:
            out["runs"] = np.array(runs)
            np.savez_compressed(os.path.join(OUT, "ref_learning", f"{scen}.npz"), **out)
            n_runs += len(runs)
    print("learning fixture:", n_runs, "runs")


def make_main_fixture():
    """The reference driver main.py, byte for byte, as a zlib blob inside a fixture (NOT a source file of this repo): the
    GPU box has no reference checkout, and tests/test_main_gpu.py must execute the UNCHANGED driver through real training
    (main.py:117-121).  The SHA-256 of the original is stored next to it."""
    import hashlib
    import zlib
    raw = open(os.path.join(REF, "main.py"), "rb").read()
    np.savez(os.path.join(OUT, "ref_main_py.npz"), blob=np.frombuffer(zlib.compress(raw, 9), np.uint8),
             sha256=np.array(hashlib.sha256(raw).hexdigest()), n_bytes=np.int64(len(raw)))
    print("main.py fixture:", len(raw), "bytes")


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    make_kat()
    make_env()
    make_methods()
    make_train_run()
    make_adversaries()
    make_learning_fixture()
    make_main_fixture()
