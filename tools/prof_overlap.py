"""CTA-budget sweep of the two big phases of the C2 update round on one GPU, the evidence behind the cost model of
rcmarl_overlap_split (csrc/train_kernels.cu, DESIGN.md 4.3):
   python tools/prof_overlap.py [budgets=148,112,96,88,80,76,72,64] [reps=3]
For every budget C, CUDA-event timings of
  - one rcmarl_grad launch (+ reduce) of the 8 cooperative full-batch jobs over 12 288 000 rows with max_ctas = C, and
  - one rcmarl_minibatch_fit call (940 SGD steps of the malicious agent's 3 chains over 131 072-row mini-batches) with
    max_ctas = C,
each phase alone on the GPU; then one epoch's worth of both (5 fit launches on the current stream, the chains on a
high-priority second stream) at the splits the cost model would consider, against the same work run one after the other.
Prints one JSON line per measurement; the least-squares fit of the model's constants at the end."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "resilient-consensus-based-marl_b200"))
import bench                                           # noqa: E402
from rcmarl import _lib as L, nets, ops                 # noqa: E402
from rcmarl.trainer import Trainer                     # noqa: E402

budgets = [int(x) for x in (sys.argv[1] if len(sys.argv) > 1 else "148,112,96,88,80,76,72,64").split(",")]
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
N, T, NA = 4096, 3000, 5
dev = torch.device("cuda:0")
sms = torch.cuda.get_device_properties(dev).multi_processor_count
try:
    smi = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem",
                                   "--format=csv,noheader", "-i", "0"], text=True).strip()
except Exception as ex:                                # noqa: BLE001
    smi = f"nvidia-smi unavailable: {ex}"
print(json.dumps(dict(device=torch.cuda.get_device_name(0), sms=sms, nvidia_smi=smi)), flush=True)

# ---- full-batch fit: 4 cooperative agents x (team-reward, critic) over the whole C2 buffer
rows_n = N * T
g = torch.Generator(device="cuda"); g.manual_seed(0)
sa = torch.randn(rows_n, 3 * NA, device=dev, generator=g)
ns = torch.randn(rows_n, 2 * NA, device=dev, generator=g)
r = torch.randn(rows_n, NA, device=dev, generator=g)
tgt = torch.randn(rows_n, device=dev, generator=g)
rs = np.random.RandomState(0)
PC, PT = L.param_count(10, 1), L.param_count(15, 1)
sums = torch.zeros(8, PT + 1, device=dev)
fit_rows = ops.make_rows(sa, ns, r, NA)
fj, keep = [], []
for j in range(8):
    kind = L.IN_SA if j % 2 == 0 else L.IN_S
    w = torch.as_tensor(nets.pack(nets.glorot_uniform(15 if kind == L.IN_SA else 10, 1, rs))).to(dev)
    keep.append(w)
    fj.append(ops.grad_job(w, tgt, sums[j] if kind == L.IN_SA else sums[j][:PC + 1], kind))
fj = (L.GradJob * 8)(*fj)
ws = ops.workspace(L.MAX_JOBS, PT)

# ---- mini-batch chains: the malicious agent of the C2 team on a filled buffer (as tools/prof_mb.py)
cfg = bench.workload("C2", N)
tr = Trainer(seed=1, **cfg)
while tr.t_filled < T:
    tr.rollout_block(min(cfg["n_ep_fixed"], (T - tr.t_filled) // cfg["max_ep_len"]))
i = cfg["labels"].index("Malicious")
tr.tdt_local[0].normal_(); tr.tdt[i].normal_(); tr.neg_r_coop.normal_()
chains = [(tr.critic_local[i], L.IN_S, tr.tdt_local[0], 1, None), (tr.tr[i], L.IN_SA, tr.neg_r_coop, 1, tr.loss_t[i:i + 1]),
          (tr.critic[i], L.IN_S, tr.tdt[i], 1, tr.loss_c[i:i + 1])]
steps = tr.mb_epochs * ((tr.t_filled + tr.mb_times - 1) // tr.mb_times)
side = torch.cuda.Stream(dev, priority=-1)


def timed(fn, n=reps):
    ts = []
    for _ in range(n + 1):                              # the first call warms up
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts[1:])), [round(t, 3) for t in ts[1:]]


def fit(c, launches=1):
    for _ in range(launches):
        ops.grad(fit_rows, fj, L.LOSS_MSE, ws, c)


def mb(c):
    tr._minibatch_sgd(chains, tr.t_filled, c)


fit_pts, mb_pts = [], []
for c in budgets:
    f_ms, f_all = timed(lambda: fit(c))
    m_ms, m_all = timed(lambda: mb(c))
    fit_pts.append((c, f_ms)); mb_pts.append((c, m_ms))
    print(json.dumps(dict(budget=c, fit_ms_per_launch=round(f_ms, 4), fit_all=f_all,
                          mb_us_per_step=round(1e3 * m_ms / steps, 3), mb_ms_per_call=round(m_ms, 3), mb_all=m_all)),
          flush=True)


def both(f):
    fork, join = torch.cuda.Event(), torch.cuda.Event()
    fork.record()
    side.wait_event(fork)
    with torch.cuda.stream(side):
        mb(sms - f)
        join.record()
    fit(f, 5)
    torch.cuda.current_stream().wait_event(join)


serial_ms, serial_all = timed(lambda: (fit(0, 5), mb(0)))
print(json.dumps(dict(epoch="serial", ms=round(serial_ms, 3), all=serial_all)), flush=True)
for f in (56, 64, 72, 80, 88):
    o_ms, o_all = timed(lambda: both(f))
    print(json.dumps(dict(epoch="overlap", fit_ctas=f, chain_ctas=sms - f, ms=round(o_ms, 3), all=o_all,
                          saved_vs_serial=round(1 - o_ms / serial_ms, 4))), flush=True)

# least-squares constants of the cost model: time = fixed + per_tile * max_j(ceil(tiles / g_j) * cost_j)
cost = {L.IN_S: 2064, L.IN_SA: 2164}                   # grad_row_cost of the critic (10 inputs) / team reward (15 inputs)


def worst(n_jobs, kinds, rows, c, balanced):
    k = (C.c_int32 * n_jobs)(*kinds)
    out = (C.c_int32 * n_jobs)()
    L.check(L.lib().rcmarl_grad_grid_plan(NA, k, n_jobs, L.LOSS_MSE, rows, int(balanced), c, out), "plan")
    tiles = (rows + 127) // 128
    return max(-(-tiles // out[j]) * cost[kinds[j]] for j in range(n_jobs))


for name, pts, n_jobs, kinds, rows, balanced, per in (
        ("fit", fit_pts, 8, [L.IN_SA, L.IN_S] * 4, rows_n, False, 1),
        ("mb", mb_pts, 3, [L.IN_S, L.IN_SA, L.IN_S], tr.mb_times * N, True, steps)):
    x = np.array([worst(n_jobs, kinds, rows, c, balanced) for c, _ in pts], float)
    y = np.array([ms * 1e6 / per for _, ms in pts], float)
    A = np.stack([np.ones_like(x), x], 1)
    (f0, f1), *_ = np.linalg.lstsq(A, y, rcond=None)
    print(json.dumps(dict(model=name, fixed_ns=round(float(f0), 1), ns_per_tile_cost=round(float(f1), 5),
                          max_rel_residual=round(float(np.max(np.abs(A @ [f0, f1] - y) / y)), 4))), flush=True)
