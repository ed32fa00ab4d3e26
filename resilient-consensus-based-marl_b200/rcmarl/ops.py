"""Thin Python wrappers over the C ABI (include/rcmarl.h): torch tensors in,
kernel launches on torch's current CUDA stream out.  PyTorch is plumbing only
(device memory, streams); every arithmetic step of the hot path happens in
librcmarl.so."""
import ctypes as C

import numpy as np
import torch

from . import _lib as L

_ws = {}


def _stream():
    return torch.cuda.current_stream().cuda_stream


def ptr(t):
    return None if t is None else t.data_ptr()


def dev_f32(x, device=None):
    """numpy / torch (any device) -> contiguous float32 CUDA tensor."""
    if isinstance(x, torch.Tensor):
        t = x
    else:
        if hasattr(x, "_t"):                       # facade Tensor
            t = x._t
        else:
            t = torch.as_tensor(np.ascontiguousarray(np.asarray(x, dtype=np.float32)))
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return t.to(device=device, dtype=torch.float32).contiguous()


def workspace(n_jobs=L.MAX_JOBS, max_params=None):
    """Persistent scratch for the *_grad / team entry points (caller-owned, no hidden allocation)."""
    dev = torch.cuda.current_device()
    if max_params is None:
        max_params = L.param_count(48, 1)
    need = L.lib().rcmarl_workspace_bytes(n_jobs, max_params)
    w = _ws.get(dev)
    if w is None or w.numel() < need:
        w = torch.empty(need, dtype=torch.uint8, device=f"cuda:{dev}")
        _ws[dev] = w
    return w


def make_rows(sa, ns, r, n_agents, row_begin=0, n_rows=None, time_idx=None, n_envs=1):
    """Build an rcmarl_rows.  Unused arrays may be None (a valid dummy pointer is passed)."""
    some = sa if sa is not None else (ns if ns is not None else r)
    R = L.Rows()
    R.sa = ptr(sa if sa is not None else some)
    R.ns = ptr(ns if ns is not None else some)
    R.r = ptr(r if r is not None else some)
    R.row_begin = int(row_begin)
    if n_rows is None:
        n_rows = (time_idx.numel() * n_envs) if time_idx is not None else some.shape[0]
    R.n_rows = int(n_rows)
    R.time_idx = ptr(time_idx)
    R.n_envs = int(n_envs)
    R.n_agents = int(n_agents)
    R._keep = (sa, ns, r, time_idx)
    return R


def clip_mean(vals, H, out=None):
    """vals: [n, P] float32 CUDA (row stride = vals.stride(0)); own = row 0."""
    n, P = vals.shape
    assert vals.stride(1) == 1
    if out is None:
        out = torch.empty(P, dtype=torch.float32, device=vals.device)
    if not (0 <= int(H) < n):
        raise L.RcmarlError(f"rcmarl_clip_mean: H={H} must satisfy 0 <= H < n={n}")
    if P == 0:
        return out
    L.check(L.lib().rcmarl_clip_mean(vals.data_ptr(), n, P, vals.stride(0), int(H), out.data_ptr(), _stream()),
            "rcmarl_clip_mean")
    return out


def value_job(out, terms, add=None, add_stride=1, add_off=0, add_scale=1.0, n_out=1, softmax=0):
    """terms: list of (weights_tensor, kind, scale)."""
    j = L.ValueJob()
    for t, (w, kind, scale) in enumerate(terms):
        j.w[t] = w.data_ptr()
        j.kind[t] = kind
        j.scale[t] = scale
    j.n_terms = len(terms)
    j.n_out = n_out
    j.softmax = softmax
    j.add = ptr(add)
    j.add_stride = add_stride
    j.add_off = add_off
    j.add_scale = add_scale
    j.out = out.data_ptr()
    j._keep = (out, terms, add)
    return j


def _arr(cls, jobs):
    a = (cls * len(jobs))(*jobs)
    return a


def values(rows, jobs):
    a = jobs if isinstance(jobs, C.Array) else _arr(L.ValueJob, jobs)
    L.check(L.lib().rcmarl_values(C.byref(rows), a, len(a), _stream()), "rcmarl_values")


def grad_job(w, target, sums, kind, action_agent=0, target_stride=1, time_idx=None):
    j = L.GradJob()
    j.w, j.target, j.sums, j.kind, j.action_agent = w.data_ptr(), target.data_ptr(), sums.data_ptr(), kind, action_agent
    j.target_stride = target_stride
    j.time_idx = ptr(time_idx)
    j._keep = (w, target, sums, time_idx)
    return j


def grad(rows, jobs, loss_mode, ws=None, max_ctas=0):
    """max_ctas > 0: plan the grid within that many CTAs (the rest of the GPU stays free for another stream)."""
    a = jobs if isinstance(jobs, C.Array) else _arr(L.GradJob, jobs)
    if ws is None:
        ws = workspace()
    L.check(L.lib().rcmarl_grad(C.byref(rows), a, len(a), loss_mode, ws.data_ptr(), ws.numel(), max_ctas, _stream()),
            "rcmarl_grad")


def sgd_job(dst, src, sums, n, coef, first=0, loss_out=None, loss_coef=0.0, loss_accumulate=0):
    j = L.SgdJob()
    j.dst, j.src, j.sums, j.loss_out = dst.data_ptr(), src.data_ptr(), sums.data_ptr(), ptr(loss_out)
    j.n, j.first, j.coef, j.loss_coef, j.loss_accumulate = n, first, coef, loss_coef, loss_accumulate
    j._keep = (dst, src, sums, loss_out)
    return j


def sgd_apply(jobs):
    a = jobs if isinstance(jobs, C.Array) else _arr(L.SgdJob, jobs)
    L.check(L.lib().rcmarl_sgd_apply(a, len(a), _stream()), "rcmarl_sgd_apply")


def minibatch_sgd(rows, gjobs, sjobs, epochs, n_times, mb_times, lr, ws=None):
    """Whole mini-batch fit (all epochs, all steps) in one library call (single GPU)."""
    ga = gjobs if isinstance(gjobs, C.Array) else _arr(L.GradJob, gjobs)
    sa = sjobs if isinstance(sjobs, C.Array) else _arr(L.SgdJob, sjobs)
    if ws is None:
        ws = workspace()
    L.check(L.lib().rcmarl_minibatch_sgd(C.byref(rows), ga, sa, len(ga), epochs, n_times, mb_times, lr, ws.data_ptr(),
                                         ws.numel(), _stream()), "rcmarl_minibatch_sgd")


class MinibatchCells:
    """Scratch of the persistent mini-batch kernel (rcmarl_minibatch_fit): zero-initialised {value, sequence} cells plus
    the host-side sequence counter (every step of every call consumes one number, never reused)."""

    def __init__(self, n_jobs=L.MAX_JOBS, max_params=None, device=None):
        if max_params is None:
            max_params = L.param_count(48, 1)
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else device
        self.buf = torch.zeros(L.lib().rcmarl_minibatch_cells_bytes(n_jobs, max_params), dtype=torch.uint8, device=dev)
        self.seq = 1


def minibatch_fit(rows, gjobs, sjobs, epochs, n_times, mb_times, lr, cells, max_ctas=0):
    """Whole mini-batch fit (all epochs, all steps, all chains) as ONE persistent kernel (csrc/minibatch_persist.cuh);
    max_ctas > 0: the chains share at most that many CTAs."""
    ga = gjobs if isinstance(gjobs, C.Array) else _arr(L.GradJob, gjobs)
    sa = sjobs if isinstance(sjobs, C.Array) else _arr(L.SgdJob, sjobs)
    steps = L.lib().rcmarl_minibatch_steps(epochs, n_times, mb_times)
    if cells.seq + steps >= 0xFFFF0000:                       # 32-bit sequence numbers: start over on clean cells
        cells.buf.zero_()
        cells.seq = 1
    L.check(L.lib().rcmarl_minibatch_fit(C.byref(rows), ga, sa, len(ga), epochs, n_times, mb_times, lr,
                                         cells.buf.data_ptr(), cells.buf.numel(), cells.seq, max_ctas, _stream()),
            "rcmarl_minibatch_fit")
    cells.seq += steps


def overlap_split(n_agents, fit_kinds, fit_rows, fit_launches, chain_kinds, mb_rows, mb_steps, world, sm_count):
    """(CTAs for the full-batch fits, CTAs for the mini-batch chains) when the two run at the same time on two streams,
    or None: run them one after the other on the whole GPU (rcmarl_overlap_split)."""
    fk = (C.c_int32 * max(len(fit_kinds), 1))(*fit_kinds)
    ck = (C.c_int32 * max(len(chain_kinds), 1))(*chain_kinds)
    out = (C.c_int32 * 2)()
    L.check(L.lib().rcmarl_overlap_split(n_agents, fk, len(fit_kinds), fit_rows, fit_launches, ck, len(chain_kinds),
                                         mb_rows, mb_steps, world, sm_count, out), "rcmarl_overlap_split")
    return (out[0], out[1]) if out[0] else None


def adam_job(theta, m, v, sums, n, grad_scale, lr_t, beta1=0.9, beta2=0.999, eps=1e-7, loss_out=None, loss_coef=0.0,
             loss_accumulate=0):
    j = L.AdamJob()
    j.theta, j.m, j.v, j.sums, j.loss_out = theta.data_ptr(), m.data_ptr(), v.data_ptr(), sums.data_ptr(), ptr(loss_out)
    j.n, j.grad_scale, j.lr_t, j.beta1, j.beta2, j.eps, j.loss_coef = n, grad_scale, lr_t, beta1, beta2, eps, loss_coef
    j.loss_accumulate = loss_accumulate
    j._keep = (theta, m, v, sums, loss_out)
    return j


def adam_apply(jobs):
    a = jobs if isinstance(jobs, C.Array) else _arr(L.AdamJob, jobs)
    L.check(L.lib().rcmarl_adam_apply(a, len(a), _stream()), "rcmarl_adam_apply")


def keras_adam_lr_t(lr, t, beta1=0.9, beta2=0.999):
    """lr_t of TF-2 Keras Adam at step t >= 1 (SURVEY Appendix A.5)."""
    return float(np.float32(lr * np.sqrt(1.0 - beta2 ** t) / (1.0 - beta1 ** t)))


def team_job(w, kind, msgs=None, msg_stride=0, in_nodes=(), H=0, sums=None, agg_out=None, agg_in=None):
    j = L.TeamJob()
    j.w, j.msgs, j.msg_stride = w.data_ptr(), ptr(msgs), msg_stride
    j.sums, j.agg_out, j.agg_in = ptr(sums), ptr(agg_out), ptr(agg_in)
    j.kind, j.n_in, j.H = kind, len(in_nodes), H
    for k, v in enumerate(in_nodes):
        j.in_nodes[k] = v
    j._keep = (w, msgs, sums, agg_out, agg_in)
    return j


def team(rows, jobs, ws=None):
    a = jobs if isinstance(jobs, C.Array) else _arr(L.TeamJob, jobs)
    if ws is None:
        ws = workspace()
    L.check(L.lib().rcmarl_team(C.byref(rows), a, len(a), ws.data_ptr(), ws.numel(), _stream()), "rcmarl_team")


def consensus_job(dst, msgs, msg_stride, n_hidden, in_nodes, H):
    j = L.ConsensusJob()
    j.dst, j.msgs, j.msg_stride, j.n_hidden, j.n_in, j.H = dst.data_ptr(), msgs.data_ptr(), msg_stride, n_hidden, len(in_nodes), H
    for k, v in enumerate(in_nodes):
        j.in_nodes[k] = v
    j._keep = (dst, msgs)
    return j


def consensus_hidden(jobs):
    a = jobs if isinstance(jobs, C.Array) else _arr(L.ConsensusJob, jobs)
    L.check(L.lib().rcmarl_consensus_hidden(a, len(a), _stream()), "rcmarl_consensus_hidden")


def reward_mix(r, agents, out=None, scale=1.0):
    """r: [rows, n_agents]; out[row] = scale * sum_k r[row, agents[k]] / len(agents) in list order."""
    n_rows, n_agents = r.shape
    if out is None:
        out = torch.empty(n_rows, dtype=torch.float32, device=r.device)
    arr = (C.c_int32 * len(agents))(*agents)
    L.check(L.lib().rcmarl_reward_mix(r.data_ptr(), n_rows, n_agents, arr, len(agents), scale, out.data_ptr(), _stream()),
            "rcmarl_reward_mix")
    return out


def state_tables(nrow, ncol, scaling=True):
    """(i - mean) / std per coordinate in float64, rounded to float32 (grid_world.py:30-35,70); mean / std are taken over
    the axis' own range, but both tables cover max(nrow, ncol) positions because the reference clips BOTH coordinates
    with nrow - 1 (grid_world.py:55), so y can leave [0, ncol) when nrow > ncol.  scaling=False: identity (the
    reference's Grid_World default)."""
    n = max(nrow, ncol)
    idx = np.arange(n)
    if not scaling:
        t = idx.astype(np.float32)
        return t, t.copy()
    x, y = np.arange(nrow), np.arange(ncol)
    tx = ((idx - np.mean(x)) / np.std(x)).astype(np.float32)
    ty = ((idx - np.mean(y)) / np.std(y)).astype(np.float32)
    return tx, ty


def rollout(actor_w, critic_w, desired, sa, ns, r, time_begin, est, ret, *, n_envs, n_agents, n_episodes, max_ep_len,
            nrow, ncol, gamma, mu=0.1, seed=0, env_offset=0, episode_offset=0, uniforms=None, init_state=None,
            scaling=True, n_active=None):
    A = L.RolloutArgs()
    A.actor_w, A.critic_w, A.desired = actor_w.data_ptr(), critic_w.data_ptr(), desired.data_ptr()
    A.sa, A.ns, A.r = sa.data_ptr(), ns.data_ptr(), r.data_ptr()
    A.time_begin = int(time_begin)
    A.est, A.ret = est.data_ptr(), ret.data_ptr()
    A.uniforms, A.init_state = ptr(uniforms), ptr(init_state)
    A.seed, A.env_offset, A.episode_offset = int(seed), int(env_offset), int(episode_offset)
    A.n_envs, A.n_agents, A.n_episodes, A.max_ep_len = n_envs, n_agents, n_episodes, max_ep_len
    A.nrow, A.ncol, A.gamma, A.mu = nrow, ncol, gamma, mu
    A.n_active = n_agents if n_active is None else int(n_active)
    if max(nrow, ncol) > L.MAX_GRID:
        raise L.RcmarlError(f"grid {nrow}x{ncol} exceeds RCMARL_MAX_GRID = {L.MAX_GRID}")
    tx, ty = state_tables(nrow, ncol, scaling)
    for i in range(len(tx)):
        A.state_tab_x[i] = float(tx[i])
        A.state_tab_y[i] = float(ty[i])
    L.check(L.lib().rcmarl_rollout(C.byref(A), _stream()), "rcmarl_rollout")


def episode_means(x, out=None):
    """x: [n_episodes, n_envs, n_agents] float32 CUDA -> [n_episodes, n_agents] means over the environments."""
    n_ep, n_envs, n_agents = x.shape
    if out is None:
        out = torch.empty(n_ep, n_agents, dtype=torch.float32, device=x.device)
    L.check(L.lib().rcmarl_episode_means(x.data_ptr(), n_ep, n_envs, n_agents, out.data_ptr(), _stream()), "rcmarl_episode_means")
    return out


def env_step(state, action, desired, nrow, reward=None):
    n_envs, n_agents = state.shape[0], state.shape[1]
    if reward is None:
        reward = torch.empty(n_envs, n_agents, dtype=torch.float32, device=state.device)
    L.check(L.lib().rcmarl_env_step(state.data_ptr(), action.data_ptr(), desired.data_ptr(), n_envs, n_agents, nrow,
                                    reward.data_ptr(), _stream()), "rcmarl_env_step")
    return reward
