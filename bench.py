#!/usr/bin/env python
"""Benchmark of the RPBCAC training hot path (BASELINE.json metric: agent-updates/sec).

  python bench.py --gpus 1 --steps K --warmup W              our arm (B200 kernels)
  python bench.py --impl reference --gpus N --steps K ...    CPU arm: the oracle port of the reference on host cores
  torchrun ... bench.py --gpus N ...                         one rank per GPU, env batch sharded (weak scaling)

A "step" is one fixed-policy block of the training loop over one batch of synthetic environments:
rollout of n_ep_fixed x max_ep_len steps for n_envs environments x n_agents agents, followed by the full
update round (Phases I-IV, training/train_agents.py:86-163) at the steady-state buffer (buffer_size + one block).
agent-updates per step = n_agents * n_envs * max_ep_len * n_ep_fixed (SURVEY 8d).

Workload (config.workload = "C2"): BASELINE.json configs[1] -- 5x5 grid, 4 cooperative + 1 malicious agent,
H = 1, 4096 parallel environments per GPU, reference hyper-parameters (main.py:31-40, slow_lr 0.002).
Inputs are larger than L2 (steady-state buffer 1.47 GB >> 126 MB), so no explicit L2 flush is needed.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
DROPIN = os.path.join(ROOT, "resilient-consensus-based-marl_b200")
for p in (ROOT, DROPIN):
    if p not in sys.path:
        sys.path.insert(0, p)

IN_NODES5 = [[0, 1, 2, 3], [1, 2, 3, 4], [2, 3, 4, 0], [3, 4, 0, 1], [4, 0, 1, 2]]
HYPER = dict(gamma=0.9, fast_lr=0.01, slow_lr=0.002, max_ep_len=20, n_ep_fixed=50, n_epochs=10, buffer_size=2000)


def load_pretrained(tag="malicious_H1_s100"):
    z = np.load(os.path.join(ROOT, "tests", "golden", "kat_est_returns.npz"))
    w = []
    for i in range(5):
        nets, n = [], 0
        while f"{tag}/agent{i}/n{n}_k0" in z.files:
            nets.append([z[f"{tag}/agent{i}/n{n}_k{k}"] for k in range(6)])
            n += 1
        w.append(nets)
    return w, z[f"{tag}/desired"], [str(x) for x in z[f"{tag}/labels"]]


def workload(name, n_envs):
    if name == "C2":
        w, desired, labels = load_pretrained()
        return dict(labels=labels, in_nodes=IN_NODES5, weights=w, desired=desired, nrow=5, ncol=5, H=1,
                    n_envs=n_envs or 4096, **HYPER)
    if name == "C1":
        w, desired, _ = load_pretrained()
        return dict(labels=["Cooperative"] * 5, in_nodes=IN_NODES5, weights=w, desired=desired, nrow=5, ncol=5, H=0,
                    n_envs=n_envs or 1, **HYPER)
    if name == "C3":
        from rcmarl import nets
        rs = np.random.RandomState(0)
        NA = 16
        w = [[nets.glorot_uniform(32, 5, rs), nets.glorot_uniform(32, 1, rs), nets.glorot_uniform(48, 1, rs)] for _ in range(NA)]
        desired = np.random.RandomState(300).randint(0, 10, size=(NA, 2))
        in_nodes = [[(i + k) % NA for k in range(6)] for i in range(NA)]
        return dict(labels=["Cooperative"] * NA, in_nodes=in_nodes, weights=w, desired=desired, nrow=10, ncol=10, H=2,
                    n_envs=n_envs or 8192, **HYPER)
    raise SystemExit(f"unknown workload {name}")


# --------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi sampled DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "200"], stdout=open(self.path, "w"),
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


def grad_traffic(workload_name):
    """dram__bytes_read.sum + dram__bytes_write.sum of one full-batch gradient launch from the committed `ncu --set full`
    capture (profiles/r02_grad_traffic.json); only valid for the workload it was captured on."""
    if workload_name != "C2":
        return None
    for name in ("r02_grad_traffic.json", "r01_grad_traffic.json"):
        try:
            return json.load(open(os.path.join(ROOT, "profiles", name)))["traffic_bytes"]
        except Exception:
            continue
    return None


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, sm_max_mhz=1965.0), "fallback"


# --------------------------------------------------------------------------------------------- CPU arm
def cpu_reference_arm(cfg, rounds, seed=0, n_envs=1, threads=None):
    """The oracle port of the reference loop (oracle/rpbcac_oracle.py) on the host cores with `n_envs` environments
    (1 = the reference's own shape; > 1 = the batched generalisation of SURVEY Appendix C that the GPU arm runs), same
    agents / hyper-parameters / schedule as the GPU arm, BLAS limited to `threads` threads (None = library default).
    Returns (agent_updates_per_s, seconds, description)."""
    if threads is not None:
        from threadpoolctl import threadpool_limits
        with threadpool_limits(limits=int(threads)):
            return cpu_reference_arm(cfg, rounds, seed, n_envs, None)
    from oracle import rpbcac_oracle as O
    labels, w = cfg["labels"], cfg["weights"]
    NA = len(labels)
    agents = []
    for i, l in enumerate(labels):
        a, c, t = w[i][0], w[i][1], w[i][2]
        if l == "Malicious":
            agents.append(O.MaliciousOracleAgent(a, c, t, cfg["slow_lr"], cfg["fast_lr"], cfg["gamma"], critic_local_w=w[i][3]))
        else:
            agents.append(O.RPBCACOracleAgent(a, c, t, cfg["slow_lr"], cfg["fast_lr"], cfg["gamma"], H=cfg["H"]))
    env = O.GridWorldOracle(cfg["nrow"], cfg["ncol"], NA, cfg["desired"], n_envs=n_envs)
    rs = np.random.RandomState(seed)
    perm_source = O.make_perm_source(seed + 1)
    n_ep, Lq = cfg["n_ep_fixed"], cfg["max_ep_len"]
    S = NS = A = R = None
    # steady-state buffer: two untimed blocks first
    def block():
        init = rs.randint(0, cfg["nrow"], size=(n_ep, n_envs, NA, 2))
        U = rs.rand(n_ep, Lq, n_envs, NA, 3).astype(np.float32)
        return O.rollout_block(env, agents, labels, n_episodes=n_ep, max_ep_len=Lq, gamma=cfg["gamma"], init_states=init, uniforms=U)
    for _ in range(2):
        s, ns, a, r, _e, _r = block()
        S, NS, A, R = (s, ns, a, r) if S is None else tuple(np.concatenate(p) for p in ((S, s), (NS, ns), (A, a), (R, r)))
    t0 = time.perf_counter()
    for _ in range(rounds):
        s, ns, a, r, _e, _r = block()
        S, NS, A, R = tuple(np.concatenate(p) for p in ((S, s), (NS, ns), (A, a), (R, r)))
        O.update_round(agents, labels, cfg["in_nodes"], S, NS, A, R, n_envs=n_envs, n_epochs=cfg["n_epochs"],
                       n_actor_steps=n_ep * Lq, common_reward=False, perm_source=perm_source)
        keep = cfg["buffer_size"] * n_envs
        S, NS, A, R = S[-keep:], NS[-keep:], A[-keep:], R[-keep:]
    dt = time.perf_counter() - t0
    upd = NA * n_envs * Lq * n_ep * rounds
    shape = "reference shape" if n_envs == 1 else "batched, SURVEY App. C"
    return upd / dt, dt, f"{rounds} update round(s) of the oracle loop at n_envs={n_envs} ({shape}), {upd} agent-updates"


# --------------------------------------------------------------------------------------------- GPU arm
_REAL_STDOUT = None
DUMP_BUFFER_ROWS = 1 << 16


def dump_outputs(out_dir, tr, est, ret, losses):
    """What the last timed step handed back (per-episode estimated and true returns, per-agent losses) and what it left
    in the trainer (the agents' packed parameters; a fixed seeded sample of the replay-buffer rows its rollout wrote),
    as out_dir/<name>.npy in float32 / float64.  The inputs are seeded, so two builds run with the same arguments can be
    compared output for output."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    n = tr.n_real
    lo, hi = (tr.t_filled - tr.block) * tr.N, tr.t_filled * tr.N
    rows = np.random.RandomState(0).choice(hi - lo, size=min(hi - lo, DUMP_BUFFER_ROWS), replace=False)
    idx = torch.as_tensor(lo + np.sort(rows), device=tr.dev)
    out = dict(est_returns=est, true_returns=ret, **losses,
               actor=tr.actor[:n], critic=tr.critic[:n], team_reward=tr.tr[:n], critic_local=tr.critic_local[:n],
               buffer_sa=tr.sa[idx], buffer_ns=tr.ns[idx], buffer_r=tr.r[idx])
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a.cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a))


def emit(line):
    """The ONE JSON line goes to the real stdout; everything else any library prints (e.g. NCCL's version banner)
    was diverted to stderr by main()."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode())
        sys.stdout.flush()


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C2")
    ap.add_argument("--n-envs", type=int, default=0, help="environments PER GPU (default: the workload's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-consensus", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (GPU arm, rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU arm's outputs; it does not apply to --impl reference")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    cfg = workload(args.workload, args.n_envs)
    NA, N = len(cfg["labels"]), cfg["n_envs"]
    upd_per_step = NA * N * cfg["max_ep_len"] * cfg["n_ep_fixed"]
    config = dict(workload=args.workload, grid=f"{cfg['nrow']}x{cfg['ncol']}", n_agents=NA, labels=cfg["labels"], H=cfg["H"],
                  n_envs_per_gpu=N, n_envs_total=N * world, steps_per_block=cfg["max_ep_len"] * cfg["n_ep_fixed"],
                  n_epochs=cfg["n_epochs"], buffer_time_rows=cfg["buffer_size"] + cfg["max_ep_len"] * cfg["n_ep_fixed"],
                  l2="inputs larger than L2 (no flush needed)", parallelism=f"dp{world}")

    if args.impl == "reference":
        if rank != 0:
            return 0
        ncores = os.cpu_count()
        # The reference is single-environment: its arm runs the oracle port at n_envs = 1 and says so in `config`
        # (the GPU arm's 4096 environments per GPU are the batched generalisation, SURVEY App. C).  One BLAS thread is the
        # fastest setting for the (<= 3000 x 20) matrices of this shape (measured: 1 / 4 / 8 threads = 1.86 / 1.11 / 1.60 k/s).
        ref_config = dict(config, n_envs_per_gpu=1, n_envs_total=1, parallelism="cpu",
                          l2="n/a (CPU arm)", note="reference shape: ONE environment; not the GPU arm's n_envs")
        vals = []
        t_all = time.perf_counter()
        for _ in range(args.steps):
            v, dt, desc = cpu_reference_arm(cfg, rounds=1, n_envs=1, threads=1)
            vals.append(v)
        v = float(np.mean(vals))
        ms_step = 1000.0 * (time.perf_counter() - t_all) / max(args.steps, 1)
        # second figure: the same oracle on a batch of environments (vectorised NumPy over rows), 8 BLAS threads
        nb = int(os.environ.get("RCMARL_CPU_BATCH_ENVS", "16"))
        bt = min(8, ncores)
        vb, dtb, descb = cpu_reference_arm(cfg, rounds=1, n_envs=nb, threads=bt)
        line = dict(metric="agent-updates/sec", value=v, unit="agent-updates/s", n_gpus=args.gpus, steps=args.steps,
                    warmup=args.warmup, ms_per_step=ms_step,
                    higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                    impl="reference", config=ref_config,
                    cpu_baseline=dict(value=v, unit="agent-updates/s", cores=1, cores_visible=ncores, kind="port",
                                      sample=desc + " per step; NumPy restatement of the reference loop, 1 BLAS thread "
                                      "(fastest for this shape) -- faster than the original TF-2.4 code path (no Keras "
                                      "retracing; the published runs imply 13-19 agent-updates/s, SURVEY 6)"),
                    cpu_batched=dict(value=vb, unit="agent-updates/s", cores=bt, n_envs=nb, seconds=dtb, sample=descb),
                    e2e=dict(value=v, unit="agent-updates/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
        emit(line)
        return 0

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from rcmarl.trainer import Trainer
    from rcmarl import ops

    tr = Trainer(rank=rank, world=world, group=group, seed=1234, **cfg)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # steady-state buffer (3 rounds in): two untimed blocks, no update
    tr.rollout_block()
    tr.rollout_block()

    def step():
        est, ret = tr.rollout_block()
        return est, ret, tr.update_round()

    for _ in range(args.warmup):
        step()
    barrier()
    tr.profile = {}
    l0 = tr.launches
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        last = step()
    e1.record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, tr, *last)
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    clk = clocks.stop() if rank == 0 else {}
    launches = tr.launches - l0
    # every rank must hold bit-identical replicated parameters after the timed region (weak scaling means nothing if the
    # replicas drifted apart): all-gather the packed parameters and compare with rank 0's
    replicas_identical = None
    if world > 1:
        mine = torch.cat([tr.actor.flatten(), tr.critic.flatten(), tr.tr.flatten(), tr.critic_local.flatten(),
                          tr.adam_m.flatten(), tr.adam_v.flatten()])
        every = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        replicas_identical = all(bool(torch.equal(every[0], e)) for e in every[1:])
        if tr.comm is not None:
            tr.comm.check()
        if not replicas_identical:
            raise SystemExit("bench.py: replicated parameters differ between ranks after the timed region")
    prof = {k: [a.elapsed_time(b) for a, b in v] for k, v in tr.profile.items()}
    tr.profile = None
    value = upd_per_step * world * args.steps / (ms / 1000.0)

    # ---- roofline of the dominant kernel: the fused fwd/bwd gradient kernel of the full-batch fits
    peaks, peak_kind = measured_peaks()
    rows = tr.t_filled * N if tr.t_filled else 0
    rows_fit = (cfg["buffer_size"] + cfg["max_ep_len"] * cfg["n_ep_fixed"]) * N
    n_coop = sum(l == "Cooperative" for l in cfg["labels"])
    fit_ms = float(np.mean(prof["fit_grad"])) if prof.get("fit_grad") else None
    roof = None
    if fit_ms:
        # SURVEY 8(d): MAC per buffer row of one fused forward + backward: critic 1 660, team reward 1 860 at 5 agents
        mac_net = lambda d: (d * 20 + 400 + 20) + (d * 20 + 840)
        d_c, d_t = 2 * NA, 3 * NA
        try:
            fp32_peak = json.load(open(os.path.join(ROOT, "profiles", "r01_fp32_peak.json")))["fp32_tflops"]
            fp32_src = ("builder-measured on this pool (FFMA2 issue-rate loop, profiles/r01_peak_rates.md); nominal "
                        "2*128*148*1.965 GHz = 74.4; MEASURED_PEAKS.json has no fp32 entry")
        except Exception:
            fp32_peak = 2 * 128 * 148 * (peaks.get("sm_max_mhz", 1965.0) * 1e6) / 1e12
            fp32_src = "nominal 2*128 lanes*148 SMs*max SM clock"
        # regime 1: the full-batch local fits (rcmarl_grad over the whole buffer, 2 nets per cooperative agent)
        alg_bytes = 20 * NA * rows_fit                       # SURVEY 8(d): 20*n_agents B per row per lock-step GD step
        flops_fit = 2.0 * n_coop * (mac_net(d_c) + mac_net(d_t)) * rows_fit
        tf_fit = flops_fit / (fit_ms * 1e-3) / 1e12
        regimes = dict(full_batch=dict(ms_per_launch=fit_ms, launches_timed=len(prof["fit_grad"]), rows=rows_fit,
                                       algorithmic_flop_per_launch=flops_fit, achieved=tf_fit, frac=tf_fit / fp32_peak))
        t_tot, f_tot = float(np.sum(prof["fit_grad"])), flops_fit * len(prof["fit_grad"])
        # regime 2: the adversaries' mini-batch chains (rcmarl_minibatch_sgd: sequential steps of mb_times x n_envs rows)
        n_mal = sum(l == "Malicious" for l in cfg["labels"])
        n_gre = sum(l == "Greedy" for l in cfg["labels"])
        mac_chain = n_mal * (2 * mac_net(d_c) + mac_net(d_t)) + n_gre * (mac_net(d_c) + mac_net(d_t))
        if prof.get("minibatch_sgd") and mac_chain:
            T_buf = rows_fit // N
            steps_call = tr.mb_epochs * ((T_buf + tr.mb_times - 1) // tr.mb_times)
            mb_ms = float(np.mean(prof["minibatch_sgd"]))
            flops_call = 2.0 * mac_chain * tr.mb_epochs * T_buf * N
            tf_mb = flops_call / (mb_ms * 1e-3) / 1e12
            regimes["mini_batch"] = dict(us_per_step=1e3 * mb_ms / steps_call, steps_per_call=steps_call,
                                         calls_timed=len(prof["minibatch_sgd"]), rows_per_step=tr.mb_times * N,
                                         algorithmic_flop_per_step=flops_call / steps_call, achieved=tf_mb,
                                         frac=tf_mb / fp32_peak)
            t_tot += float(np.sum(prof["minibatch_sgd"]))
            f_tot += flops_call * len(prof["minibatch_sgd"])
        tf_w = f_tot / (t_tot * 1e-3) / 1e12
        kname = ("grad_kernel_ws + mb_persist_ws_kernel (warp-specialised tcgen05 3xTF32 + FFMA2 fused MLP forward/backward; "
                 "rcmarl_grad + rcmarl_minibatch_fit)") if tr.NA == 5 else \
            f"grad_kernel<{tr.NA},MSE> (FFMA2 fused MLP forward/backward; rcmarl_grad + rcmarl_minibatch_fit)"
        roof = dict(kernel=kname,
                    bound="fp32", achieved=tf_w, peak=fp32_peak, unit="TFLOP/s", frac=tf_w / fp32_peak,
                    frac_is="time-weighted over both regimes of the kernel (full-batch fits + mini-batch chains)",
                    share_of_step=t_tot / ms, traffic=grad_traffic(args.workload),
                    traffic_note="DRAM bytes of ONE full-batch launch (ncu --set full); compare with hbm_view.algorithmic_bytes_per_launch",
                    peak_source=fp32_src, regimes=regimes,
                    hbm_view=dict(achieved=alg_bytes / (fit_ms * 1e-3) / 1e9, peak=peaks["hbm_gbs"], unit="GB/s",
                                  frac=alg_bytes / (fit_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                  algorithmic_bytes_per_launch=alg_bytes,
                                  peak_source=f"{peak_kind} (MEASURED_PEAKS.json hbm_gbs)",
                                  note="full-batch launch; the kernel is FP32-FMA bound (350 FLOP/B), this view is for the record"))
    breakdown = {k: dict(ms_total=float(np.sum(v)), calls=len(v)) for k, v in prof.items()}

    # ---- consensus microbench (BASELINE metric part 2, C5): 64 x 1M clip-mean, HBM-bound
    cons = None
    if rank == 0 and not args.no_consensus:
        g = torch.Generator(device="cuda")
        g.manual_seed(0)
        # three rotating inputs of 272 MB each: every launch reads data that the 126 MB L2 cannot still hold
        Xs = [torch.randn(64, 1 << 20, device="cuda", generator=g) for _ in range(3)]
        out = torch.empty(1 << 20, device="cuda")
        cons = {}
        reps = 12
        for H in (0, 1, 2, 4):
            for i in range(3):
                ops.clip_mean(Xs[i], H, out)
            ts = []
            for _ in range(5):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for i in range(reps):
                    ops.clip_mean(Xs[i % 3], H, out)
                b.record()
                torch.cuda.synchronize()
                ts.append(a.elapsed_time(b) / reps)
            t = float(np.median(ts))
            gbs = 4.0 * (1 << 20) * 65 / (t * 1e-3) / 1e9
            cons[f"H={H}"] = dict(ms=t, achieved=gbs, unit="GB/s", frac=gbs / peaks["hbm_gbs"])
        cons["algorithmic_bytes"] = 4 * (1 << 20) * 65
        cons["peak"] = peaks["hbm_gbs"]
        cons["l2"] = "12 back-to-back launches over 3 rotating 272 MB inputs (each larger than L2), CUDA events around the 12"
        del Xs

    # ---- e2e: the reference-facing API (training.train_agents.train_RPBCAC) with HOST buffers
    e2e = None
    if not args.no_e2e:
        barrier()                                             # ranks enter the end-to-end arm together
        e2e = e2e_arm(cfg, args, rank, world, tr)

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        v, dt, desc = cpu_reference_arm(cfg, rounds=2, n_envs=1, threads=1)
        nb, bt = int(os.environ.get("RCMARL_CPU_BATCH_ENVS", "16")), min(8, os.cpu_count())
        vb, dtb, descb = cpu_reference_arm(cfg, rounds=1, n_envs=nb, threads=bt)
        cpu = dict(value=v, unit="agent-updates/s", cores=1, cores_visible=os.cpu_count(), kind="port", seconds=dt,
                   sample=desc + "; NumPy restatement of the reference loop (oracle/rpbcac_oracle.py), 1 BLAS thread (fastest "
                   "for the reference's (<= 3000 x 20) matrices); faster than the original TF-2.4 path",
                   batched=dict(value=vb, unit="agent-updates/s", cores=bt, n_envs=nb, seconds=dtb, sample=descb))

    if rank == 0:
        line = dict(metric="agent-updates/sec", value=value, unit="agent-updates/s", n_gpus=world, steps=args.steps,
                    warmup=args.warmup, ms_per_step=ms / args.steps, higher_is_better=True, scaling="weak",
                    vs_baseline=None, dtype="f32", data="synthetic", config=config, clocks=clk, e2e=e2e,
                    gpu_launches=launches, replicas_identical=replicas_identical, roofline=roof, consensus_roofline=cons, cpu_baseline=cpu,
                    breakdown_ms=breakdown, update_rounds_per_s=args.steps / (ms / 1000.0))
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


def e2e_arm(cfg, args, rank, world, tr):
    """Same metric through the public, reference-shaped API with HOST buffers: agents are built from host (NumPy)
    weights, the steady-state replay buffer is handed over as host arrays (exp_buffer, train_agents.py:36-40),
    train_RPBCAC runs `steps` blocks and returns host weights + the sim_data frame.  Host->device copies of the
    buffer / weights / permutations and device->host reads of logs, losses and weights are inside the timed region."""
    import torch
    try:
        from rcmarl import api
    except Exception as ex:                                   # pragma: no cover
        return dict(value=None, unit="agent-updates/s", error=f"public API unavailable: {ex!r}")
    NA, N = len(cfg["labels"]), cfg["n_envs"]
    keep = cfg["buffer_size"] * N
    host = api.export_buffer(tr, keep)                        # pinned host copies of the newest buffer_size time rows
    n_steps = args.steps
    res = api.timed_train(cfg, host, n_blocks=n_steps, rank=rank, world=world)
    upd = NA * N * cfg["max_ep_len"] * cfg["n_ep_fixed"] * n_steps * world
    return dict(value=upd / res["seconds"], unit="agent-updates/s", h2d_bytes_per_step=res["h2d_bytes"] // n_steps,
                d2h_bytes_per_step=res["d2h_bytes"] // n_steps, seconds=res["seconds"],
                api="training.train_agents.train_RPBCAC(env, agents, args, exp_buffer=host arrays)")


if __name__ == "__main__":
    sys.exit(main())
