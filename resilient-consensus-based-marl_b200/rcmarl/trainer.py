"""Batched RPBCAC training engine (device-resident; one process per GPU).

Restates training/train_agents.py:46-163 for N independent environments that
share one set of agents (SURVEY Appendix C): the replay buffer is one
time-major tensor in HBM, the rollout of a whole fixed-policy block is ONE
kernel, and every phase of the update round is a handful of fused launches
over all agents (csrc/, C ABI in include/rcmarl.h).  With n_envs == 1 and
injected randomness it reproduces the reference update for update.

Data-parallel (SURVEY 8e): each rank owns n_envs environments and their buffer
rows for ever; parameters are replicated; the only exchange is one all-reduce
of the packed UNSCALED gradient sums per SGD / Adam / projection step.
"""
import os

import numpy as np
import torch

from . import _lib as L
from . import dist_util, nets, ops

COOP, GREEDY, MALICIOUS, FAULTY = "Cooperative", "Greedy", "Malicious", "Faulty"
PAD = "(unused agent slot)"


class Trainer:
    def __init__(self, *, labels, in_nodes, weights, desired, n_envs=1, nrow=5, ncol=5, gamma=0.9, H=0,
                 fast_lr=0.01, slow_lr=0.01, max_ep_len=20, n_ep_fixed=50, n_epochs=10, buffer_size=2000,
                 common_reward=False, mu=0.1, seed=0, device=None, rank=0, world=1, group=None,
                 perm_source=None, local_steps=5, mb_epochs=10, mb_times=32, actor_mb_times=200,
                 capacity_times=None, adam_state=None, scaling=True, fixed_initial_state=None):
        L.lib()
        # Any team size up to 16 (main.py:26): the kernels are instantiated for 5 and 16 agents, a team of n_real agents
        # runs on the next instantiation with the extra agent slots zero (inputs and W1 rows, rcmarl/nets.py) -- exactly the
        # n_real-agent problem.  self.NA is the kernel instantiation, self.n_real the team.
        self.n_real = len(labels)
        try:
            NA = nets.kernel_agents(self.n_real)
        except ValueError as ex:
            raise L.RcmarlError(str(ex))
        self.NA = NA
        self.labels = list(labels) + [PAD] * (NA - self.n_real)
        self.in_nodes = [list(x) for x in in_nodes]
        self.coop = [i for i, l in enumerate(self.labels) if l == COOP]
        self.N, self.nrow, self.ncol = int(n_envs), int(nrow), int(ncol)
        self.gamma, self.mu = float(gamma), float(mu)
        # per-agent trimming parameter H and fast learning rate (agents/resilient_CAC_agents.py:28-36 stores both per agent)
        n_real = self.n_real
        self.H = [int(H)] * n_real if np.isscalar(H) else [int(x) for x in H]
        self.fast_lr = [float(fast_lr)] * n_real if np.isscalar(fast_lr) else [float(x) for x in fast_lr]
        if len(self.H) != n_real or len(self.fast_lr) != n_real:
            raise L.RcmarlError("H / fast_lr must be scalars or one value per agent")
        self.H += [0] * (NA - n_real)
        self.fast_lr += [self.fast_lr[0]] * (NA - n_real)
        self.slow_lr = [float(slow_lr)] * NA if np.isscalar(slow_lr) else [float(x) for x in slow_lr] + [0.0] * (NA - n_real)
        self.max_ep_len, self.n_ep_fixed, self.n_epochs = int(max_ep_len), int(n_ep_fixed), int(n_epochs)
        self.block = self.max_ep_len * self.n_ep_fixed                    # time rows per fixed-policy block
        self.buffer_size = int(buffer_size)                               # in time rows (train_agents.py:158)
        self.common_reward = bool(common_reward)
        self.seed, self.rank, self.world, self.group = int(seed), int(rank), int(world), group
        self.local_steps, self.mb_epochs = int(local_steps), int(mb_epochs)
        self.mb_times, self.actor_mb_times = int(mb_times), int(actor_mb_times)
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.perm_source = perm_source
        self._perm_gen = torch.Generator(device="cpu")
        self._perm_gen.manual_seed(self.seed * 7919 + 17)
        self.episodes_done = 0
        # Grid_World(scaling=..., randomize_state=False, initial_state=...) of the reference (grid_world.py:21-45)
        self.scaling = bool(scaling)
        self.fixed_initial_state = None if fixed_initial_state is None else np.asarray(fixed_initial_state, np.int32).reshape(NA, 2)
        self._fixed_init_dev = None

        self.PA, self.PC, self.PT = L.param_count(2 * NA, 5), L.param_count(2 * NA, 1), L.param_count(3 * NA, 1)
        f32 = dict(dtype=torch.float32, device=self.dev)
        self.actor = torch.zeros(NA, self.PA, **f32)
        self.critic = torch.zeros(NA, self.PC, **f32)
        self.tr = torch.zeros(NA, self.PT, **f32)
        self.critic_local = torch.zeros(NA, self.PC, **f32)
        for i, w in enumerate(weights):
            self.actor[i].copy_(torch.as_tensor(nets.pack_padded(w[0], 2 * NA)))
            self.critic[i].copy_(torch.as_tensor(nets.pack_padded(w[1], 2 * NA)))
            self.tr[i].copy_(torch.as_tensor(nets.pack_padded(w[2], 3 * NA)))
            self.critic_local[i].copy_(torch.as_tensor(nets.pack_padded(w[3] if len(w) > 3 else w[1], 2 * NA)))
        self.msg_c = torch.zeros(NA, self.PC, **f32)
        self.msg_t = torch.zeros(NA, self.PT, **f32)
        self.adam_m = torch.zeros(NA, self.PA, **f32)
        self.adam_v = torch.zeros(NA, self.PA, **f32)
        self.adam_t = [0] * NA
        if adam_state is not None:
            for i, st in enumerate(adam_state):
                if st is not None:
                    self.adam_m[i].copy_(st[0]); self.adam_v[i].copy_(st[1]); self.adam_t[i] = int(st[2])
        des = np.zeros((NA, 2), np.int32)
        des[:self.n_real] = np.asarray(desired, np.int32).reshape(self.n_real, 2)
        self.desired = torch.as_tensor(des).to(self.dev)

        # replay buffer (time-major, row = t * N + e); capacity = buffer_size + one block
        self.Tcap = int(capacity_times) if capacity_times else self.buffer_size + self.block
        rows = self.Tcap * self.N
        self.sa = torch.zeros(rows, 3 * NA, **f32)
        self.ns = torch.zeros(rows, 2 * NA, **f32)
        self.r = torch.zeros(rows, NA, **f32)
        self.t_filled = 0
        # per-row scratch
        self.tdt = torch.zeros(NA, rows, **f32)          # critic TD targets (train_agents.py / res..py:114-115)
        n_mal = sum(l == MALICIOUS for l in self.labels)
        self.tdt_local = torch.zeros(max(n_mal, 1), rows if n_mal else 1, **f32)
        self.delta = torch.zeros(NA, rows, **f32)        # TD errors (actor window), indexed by absolute buffer row
        self.r_coop = torch.zeros(rows, **f32)
        self.neg_r_coop = torch.zeros(rows if n_mal else 1, **f32)
        # reduction outputs (contiguous so that one all-reduce covers a whole launch)
        self.sums_fit = torch.zeros(2 * NA, self.PT + 1, **f32)
        self.sums_mb = torch.zeros(3 * NA, self.PT + 1, **f32)
        self.sums_team = torch.zeros(2 * NA, 22, **f32)
        self.sums_actor = torch.zeros(NA, self.PA + 1, **f32)
        self.loss_c = torch.zeros(NA, **f32)
        self.loss_t = torch.zeros(NA, **f32)
        self.loss_a = torch.zeros(NA, **f32)
        self.ws = ops.workspace(L.MAX_JOBS, self.PT if NA == 5 else L.param_count(48, 1))
        # persistent mini-batch kernel (rcmarl_minibatch_fit); RCMARL_MB_PERSIST=0 selects the round-1 launch chain
        self.mb_cells = None
        if os.environ.get("RCMARL_MB_PERSIST", "1") != "0":
            self.mb_cells = ops.MinibatchCells(L.MAX_JOBS, self.PT if NA == 5 else L.param_count(48, 1), self.dev)
        self._side = None                                 # stream of the mini-batch chains when they overlap the fits
        self.launches = 0                                 # kernels launched by this engine (bench: gpu_launches)
        self.profile = None                               # bench.py: {"fit_grad": [(start_evt, end_evt), ...], ...}
        self.h2d_bytes = 4 * sum(x.numel() for x in (self.actor, self.critic, self.tr, self.critic_local))
        self.d2h_bytes = 0
        # data parallel: exchange gradient sums inside the reduction kernels over NVLink peer memory (csrc/comm.cuh);
        # RCMARL_PEER_COMM=0 selects one NCCL all-reduce per step instead
        self.comm = None
        if self.world > 1 and os.environ.get("RCMARL_PEER_COMM", "1") != "0":
            self.comm = self._try_peer_comm()

    # ------------------------------------------------------------------ helpers
    def _try_peer_comm(self):
        """Set up the peer-memory exchange on every rank, or on none: the ranks agree (MIN all-reduce of a success
        flag) so that a box without IPC / peer access falls back to the NCCL path consistently instead of deadlocking."""
        import torch.distributed as dist
        from .comm import PeerComm
        comm, ok = None, 1
        try:
            comm = PeerComm(self.rank, self.world, self.group)
        except Exception as ex:                                      # noqa: BLE001 -- any failure means "use NCCL"
            ok = 0
            if self.rank == 0:
                print(f"[rcmarl] peer-memory exchange unavailable ({ex}); using NCCL all-reduce", flush=True)
        flag = torch.tensor([ok], device=self.dev, dtype=torch.int32)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
        if int(flag.item()) == 0:
            if comm is not None:
                comm.close()
            return None
        return comm

    def _allreduce(self, t):
        """Sum the packed gradient sums over ranks -- unless the bound peer-memory context already did it in-kernel."""
        if self.comm is not None:
            return t
        return dist_util.allreduce_sums(t, self.world, self.group)

    def _timed(self, name, fn, *args):
        """Run fn(*args); when profiling is on, bracket it with CUDA events on the launching stream."""
        if self.profile is None:
            return fn(*args)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn(*args)
        b.record()
        self.profile.setdefault(name, []).append((a, b))

    def _perm(self, T):
        if self.perm_source is not None:
            p = np.asarray(self.perm_source(T), np.int32)
            assert p.shape == (T,)
            return torch.as_tensor(p)
        return torch.randperm(T, generator=self._perm_gen, dtype=torch.int32)

    def _rows(self, row_begin, n_rows, time_idx=None):
        return ops.make_rows(self.sa, self.ns, self.r, self.NA, row_begin, n_rows, time_idx, self.N)

    def get_weights(self, i):
        """[actor, critic, TR(, critic_local)] as Keras weight lists (get_parameters, res..py:221-223)."""
        NA, n = self.NA, self.n_real
        self.d2h_bytes += 4 * (self.PA + self.PC + self.PT + (self.PC if self.labels[i] == MALICIOUS else 0))
        out = [nets.unpack_padded(self.actor[i].cpu().numpy(), 2 * n, 2 * NA, 5),
               nets.unpack_padded(self.critic[i].cpu().numpy(), 2 * n, 2 * NA, 1),
               nets.unpack_padded(self.tr[i].cpu().numpy(), 3 * n, 3 * NA, 1)]
        if self.labels[i] == MALICIOUS:
            out.append(nets.unpack_padded(self.critic_local[i].cpu().numpy(), 2 * n, 2 * NA, 1))
        return out

    # ------------------------------------------------------------------ rollout
    def rollout_block(self, n_episodes=None, uniforms=None, init_state=None):
        """Episodes under the current (fixed) policy for all environments: ONE kernel launch
        (train_agents.py:46-80).  Returns per-episode means over this rank's environments:
        est[n_ep, NA] (critic(state_0), :60-62) and ret[n_ep, NA] (discounted returns, :71)."""
        n_ep = self.n_ep_fixed if n_episodes is None else int(n_episodes)
        Lq = self.max_ep_len
        if self.t_filled + n_ep * Lq > self.Tcap:
            raise L.RcmarlError("replay buffer overflow: call update_round() (which trims) before the next block")
        est = torch.empty(n_ep, self.N, self.NA, dtype=torch.float32, device=self.dev)
        ret = torch.empty(n_ep, self.N, self.NA, dtype=torch.float32, device=self.dev)
        self._timed("rollout", self._rollout_launch, est, ret, n_ep, uniforms, init_state)
        self.launches += 1
        self.t_filled += n_ep * Lq
        self.episodes_done += n_ep
        stats = torch.empty(2, n_ep, self.NA, dtype=torch.float32, device=self.dev)
        ops.episode_means(est, stats[0])                                   # logging only (train_agents.py:168-180)
        ops.episode_means(ret, stats[1])
        self.launches += 2
        if self.world > 1:
            dist_util.allreduce_sums(stats, self.world, self.group)     # logging only (NCCL)
            stats /= self.world
        stats = stats.cpu().numpy()[:, :, :self.n_real]
        self.d2h_bytes += stats.nbytes
        return stats[0], stats[1]

    def _rollout_launch(self, est, ret, n_ep, uniforms, init_state):
        Lq = self.max_ep_len
        if init_state is None and self.fixed_initial_state is not None:    # randomize_state=False: every reset -> initial_state
            if self._fixed_init_dev is None or self._fixed_init_dev.shape[0] < n_ep:
                host = np.broadcast_to(self.fixed_initial_state, (n_ep, self.N, self.NA, 2))
                self._fixed_init_dev = torch.as_tensor(np.ascontiguousarray(host)).to(self.dev)
            init_state = self._fixed_init_dev
        ops.rollout(self.actor, self.critic, self.desired, self.sa, self.ns, self.r, self.t_filled, est, ret,
                    n_envs=self.N, n_agents=self.NA, n_episodes=n_ep, max_ep_len=Lq, nrow=self.nrow, ncol=self.ncol,
                    n_active=self.n_real, gamma=self.gamma, mu=self.mu, seed=self.seed, env_offset=self.rank * self.N,
                    episode_offset=self.episodes_done, uniforms=uniforms, init_state=init_state, scaling=self.scaling)

    def load_rows(self, s, ns, a, r):
        """Append externally produced transitions (exp_buffer, train_agents.py:36-40; parity tests; bench e2e).
        s, ns: (B, NA, 2); a, r: (B, NA, 1) as lists / NumPy arrays / (pinned) host or device torch tensors;
        B must be a multiple of n_envs, rows time-major.  The sa = concat([s, a]) of train_agents.py:93 is formed by
        strided device copies (data movement only)."""
        n = self.n_real

        def t(x, last):
            if not isinstance(x, torch.Tensor):
                x = torch.as_tensor(np.asarray(x, np.float32))
            return x.reshape(-1, n, last)
        s, ns, a, r = t(s, 2), t(ns, 2), t(a, 1), t(r, 1)
        B = s.shape[0]
        assert B % self.N == 0 and self.t_filled * self.N + B <= self.Tcap * self.N
        o = self.t_filled * self.N
        sa3 = self.sa.view(-1, self.NA, 3)                      # unused agent slots stay zero (the buffers start zeroed)
        sa3[o:o + B, :n, :2].copy_(s.to(self.dev, dtype=torch.float32, non_blocking=True))
        sa3[o:o + B, :n, 2:].copy_(a.to(self.dev, dtype=torch.float32, non_blocking=True))
        self.ns.view(-1, self.NA, 2)[o:o + B, :n].copy_(ns.to(self.dev, dtype=torch.float32, non_blocking=True))
        self.r.view(-1, self.NA, 1)[o:o + B, :n].copy_(r.to(self.dev, dtype=torch.float32, non_blocking=True))
        self.h2d_bytes += 4 * B * n * 6
        self.t_filled += B // self.N

    # ------------------------------------------------------------------ update round
    def update_round(self):
        """training/train_agents.py:86-163 for all agents and all local environments."""
        NA, N, T = self.NA, self.N, self.t_filled
        B = T * N
        Bg = B * self.world
        lab = self.labels
        coop = self.coop
        mal = [i for i in range(NA) if lab[i] == MALICIOUS]
        rows_all = self._rows(0, B)
        r_col = [self.r[:, i] for i in range(NA)]

        if coop:                                                           # :96-98
            ops.reward_mix(self.r[:B], coop, out=self.r_coop, scale=1.0)
            self.launches += 1
            if mal:
                ops.reward_mix(self.r[:B], coop, out=self.neg_r_coop, scale=-1.0)
                self.launches += 1

        def applied(i):                                                    # r_applied, :106
            return (self.r_coop, 1) if self.common_reward else (r_col[i], NA)

        # ---- job tables that do not change across epochs
        td_jobs = []
        for i in range(NA):
            if lab[i] == COOP:
                add, st = applied(i)
                td_jobs.append(ops.value_job(self.tdt[i], [(self.critic[i], L.IN_NS, self.gamma)], add=add, add_stride=st))
            elif lab[i] == GREEDY:
                td_jobs.append(ops.value_job(self.tdt[i], [(self.critic[i], L.IN_NS, self.gamma)], add=r_col[i], add_stride=NA))
            elif lab[i] == MALICIOUS:
                k = mal.index(i)
                td_jobs.append(ops.value_job(self.tdt_local[k], [(self.critic_local[i], L.IN_NS, self.gamma)],
                                             add=r_col[i], add_stride=NA))                       # adversarial:148-149
                td_jobs.append(ops.value_job(self.tdt[i], [(self.critic[i], L.IN_NS, self.gamma)],
                                             add=self.neg_r_coop, add_stride=1))                 # adversarial:131-132
        td_arr = (L.ValueJob * len(td_jobs))(*td_jobs) if td_jobs else None

        fit_first, fit_next, fit_apply_first, fit_apply_next = [], [], [], []
        for n, i in enumerate(coop):
            lr2 = self.fast_lr[i] * 2.0 / Bg
            tgt_t, st_t = applied(i)
            sc, stt = self.sums_fit[2 * n][:self.PC + 1], self.sums_fit[2 * n + 1]
            for first in (True, False):
                wc = self.critic[i] if first else self.msg_c[i]
                wt = self.tr[i] if first else self.msg_t[i]
                gj = [ops.grad_job(wt, tgt_t, stt, L.IN_SA, target_stride=st_t),
                      ops.grad_job(wc, self.tdt[i], sc, L.IN_S)]
                aj = [ops.sgd_job(self.msg_t[i], wt, stt, self.PT, lr2, loss_out=self.loss_t[i:i + 1] if first else None,
                                  loss_coef=1.0 / Bg),
                      ops.sgd_job(self.msg_c[i], wc, sc, self.PC, lr2, loss_out=self.loss_c[i:i + 1] if first else None,
                                  loss_coef=1.0 / Bg)]
                (fit_first if first else fit_next).extend(gj)
                (fit_apply_first if first else fit_apply_next).extend(aj)
        arr = lambda cls, js: (cls * len(js))(*js) if js else None
        fit_first, fit_next = arr(L.GradJob, fit_first), arr(L.GradJob, fit_next)
        fit_apply_first, fit_apply_next = arr(L.SgdJob, fit_apply_first), arr(L.SgdJob, fit_apply_next)

        # mini-batch chains of the adversaries (adversarial:133,150,163,239,251), node order = permutation order
        chains = []                                       # (weights in place, kind, target, stride, loss slot, lr)
        for i in range(NA):
            lr_i = self.fast_lr[i]
            if lab[i] == MALICIOUS:
                k = mal.index(i)
                chains.append((self.critic_local[i], L.IN_S, self.tdt_local[k], 1, None, lr_i))
                chains.append((self.tr[i], L.IN_SA, self.neg_r_coop, 1, self.loss_t[i:i + 1], lr_i))
                chains.append((self.critic[i], L.IN_S, self.tdt[i], 1, self.loss_c[i:i + 1], lr_i))
            elif lab[i] == GREEDY:
                chains.append((self.tr[i], L.IN_SA, r_col[i], NA, self.loss_t[i:i + 1], lr_i))
                chains.append((self.critic[i], L.IN_S, self.tdt[i], 1, self.loss_c[i:i + 1], lr_i))

        # The chains and the cooperative fits touch disjoint parameters and scratch and only read the buffer and the TD
        # targets, so they may run at the same time on two streams, each on its share of the SMs (rcmarl_overlap_split).
        fit_ctas = mb_ctas = 0
        if coop and chains and self.mb_cells is not None:
            split = ops.overlap_split(NA, [j.kind for j in fit_first], B, self.local_steps, [ch[1] for ch in chains],
                                      self.mb_times * N, self.mb_epochs * ((T + self.mb_times - 1) // self.mb_times),
                                      self.world, torch.cuda.get_device_properties(self.dev).multi_processor_count)
            if split is not None:
                fit_ctas, mb_ctas = split
                if self._side is None:
                    self._side = torch.cuda.Stream(self.dev, priority=-1)

        cons_jobs, team_jobs, team_apply = [], [], []
        for n, i in enumerate(coop):
            nodes = self.in_nodes[i]
            cons_jobs.append(ops.consensus_job(self.critic[i], self.msg_c, self.PC, nets.n_hidden_params(2 * NA), nodes, self.H[i]))
            cons_jobs.append(ops.consensus_job(self.tr[i], self.msg_t, self.PT, nets.n_hidden_params(3 * NA), nodes, self.H[i]))
            team_jobs.append(ops.team_job(self.critic[i], L.IN_S, self.msg_c, self.PC, nodes, self.H[i], sums=self.sums_team[2 * n]))
            team_jobs.append(ops.team_job(self.tr[i], L.IN_SA, self.msg_t, self.PT, nodes, self.H[i], sums=self.sums_team[2 * n + 1]))
            team_apply.append(ops.sgd_job(self.critic[i], self.critic[i], self.sums_team[2 * n], self.PC, -1.0 / Bg, first=self.PC - 21))
            team_apply.append(ops.sgd_job(self.tr[i], self.tr[i], self.sums_team[2 * n + 1], self.PT, -1.0 / Bg, first=self.PT - 21))
        cons_jobs, team_jobs, team_apply = arr(L.ConsensusJob, cons_jobs), arr(L.TeamJob, team_jobs), arr(L.SgdJob, team_apply)

        for _epoch in range(self.n_epochs):                                # :100
            # ---------------- I) local updates (:105-121)
            if td_arr is not None:
                ops.values(rows_all, td_arr)
                self.launches += 1
            if mb_ctas:                                                    # chains first: the side stream has priority
                fork, join = torch.cuda.Event(), torch.cuda.Event()
                fork.record()
                self._side.wait_event(fork)
                with torch.cuda.stream(self._side):                        # perms are allocated on this stream
                    self._timed("minibatch_sgd", self._minibatch_sgd, chains, T, mb_ctas)
                    join.record()
            if coop:
                for step in range(self.local_steps):                      # fit(batch_size=B, epochs=5), res..py:118,136
                    self._timed("fit_grad", ops.grad, rows_all, fit_first if step == 0 else fit_next, L.LOSS_MSE, self.ws,
                                fit_ctas)
                    self._allreduce(self.sums_fit[:2 * len(coop)])
                    ops.sgd_apply(fit_apply_first if step == 0 else fit_apply_next)
                    self.launches += 3
            if mb_ctas:
                torch.cuda.current_stream().wait_event(join)
            elif chains:
                self._timed("minibatch_sgd", self._minibatch_sgd, chains, T)
            for i in range(self.n_real):                                   # the transmitted messages (:118-121)
                if lab[i] != COOP:
                    self.msg_c[i].copy_(self.critic[i])
                    self.msg_t[i].copy_(self.tr[i])
            # ---------------- II) resilient consensus (:125-145)
            if coop:
                ops.consensus_hidden(cons_jobs)
                self._timed("team", ops.team, rows_all, team_jobs, self.ws)
                self._allreduce(self.sums_team[:2 * len(coop)])
                ops.sgd_apply(team_apply)
                # consensus_hidden + team_kernel per input kind (critic / team-reward nets) + reduce + sgd
                self.launches += 3 + len({j.kind for j in team_jobs})

        # ---------------- III) actor updates (:149-153) on the newest block
        Ta = min(self.block, T)
        a0 = (T - Ta) * N
        rows_act = self._rows(a0, Ta * N)
        d_jobs = []
        for i in range(self.n_real):
            if lab[i] == COOP:                                             # res..py:95-98
                d_jobs.append(ops.value_job(self.delta[i], [(self.tr[i], L.IN_SA, 1.0), (self.critic[i], L.IN_NS, self.gamma),
                                                            (self.critic[i], L.IN_S, -1.0)]))
            else:                                                          # adversarial:38-40,113-115,221-223
                cw = self.critic_local[i] if lab[i] == MALICIOUS else self.critic[i]
                d_jobs.append(ops.value_job(self.delta[i], [(cw, L.IN_NS, self.gamma), (cw, L.IN_S, -1.0)],
                                            add=r_col[i], add_stride=NA))
        ops.values(rows_act, arr(L.ValueJob, d_jobs))
        self.launches += 1
        Bag = Ta * N * self.world
        if coop:
            gj, aj = [], []
            for n, i in enumerate(coop):
                self.adam_t[i] += 1
                gj.append(ops.grad_job(self.actor[i], self.delta[i], self.sums_actor[n], L.IN_S, action_agent=i))
                aj.append(ops.adam_job(self.actor[i], self.adam_m[i], self.adam_v[i], self.sums_actor[n], self.PA, 1.0 / Bag,
                                       ops.keras_adam_lr_t(self.slow_lr[i], self.adam_t[i]), loss_out=self.loss_a[i:i + 1],
                                       loss_coef=1.0 / Bag))
            ops.grad(rows_act, arr(L.GradJob, gj), L.LOSS_CE, self.ws)
            self._allreduce(self.sums_actor[:len(coop)])
            ops.adam_apply(arr(L.AdamJob, aj))
            self.launches += 3
        adv = [i for i in range(self.n_real) if lab[i] != COOP]
        if adv:
            self._minibatch_adam(adv, T, Ta, a0)

        n = self.n_real
        losses = dict(critic_loss=self.loss_c.cpu().numpy().astype(np.float64)[:n],
                      TR_loss=self.loss_t.cpu().numpy().astype(np.float64)[:n],
                      actor_loss=self.loss_a.cpu().numpy().astype(np.float64)[:n])
        self.d2h_bytes += 3 * 8 * NA
        # ---------------- IV) buffer trim (:158-163)
        self.trim()
        return losses

    def _minibatch_sgd(self, chains, T, max_ctas=0):
        """10 epochs x ceil(T/32) sequential SGD steps per chain; a mini-batch = 32 time rows x all environments
        (Appendix C).  All chains advance in lock-step: one grad launch + one apply launch per step."""
        N, nb = self.N, (T + self.mb_times - 1) // self.mb_times
        E = self.mb_epochs
        perms = torch.stack([torch.stack([self._perm(T) for _ in range(E)]) for _ in chains]).to(self.dev)  # [C,E,T]
        self.h2d_bytes += 4 * perms.numel()
        base = perms.data_ptr()
        gj, aj = [], []
        lrs = [ch[5] if len(ch) > 5 else self.fast_lr[0] for ch in chains]
        for c, (w, kind, tgt, st, loss) in enumerate([ch[:5] for ch in chains]):
            n = self.PT if kind == L.IN_SA else self.PC
            sums = self.sums_mb[c][:n + 1]
            gj.append(ops.grad_job(w, tgt, sums, kind, target_stride=st, time_idx=perms))
            persistent = self.mb_cells is not None and (self.world == 1 or self.comm is not None)
            aj.append(ops.sgd_job(w, w, sums, n, 0.0, loss_out=loss, loss_coef=1.0 / (T * N * self.world),
                                  loss_accumulate=0 if persistent else 1))     # the persistent kernel writes the epoch-0 loss once
            if loss is not None and not persistent:
                loss.zero_()
        gj, aj = (L.GradJob * len(gj))(*gj), (L.SgdJob * len(aj))(*aj)
        rows = self._rows(0, 0, perms)
        nC = len(chains)
        nb_steps = E * nb
        if self.world == 1 or self.comm is not None:       # whole fit in one library call (fused reduce [+ exchange] + apply)
            for c in range(nC):
                gj[c].time_idx = base + 4 * (c * E * T)
            if self.mb_cells is not None:                   # one persistent kernel for the whole fit
                for c in range(nC):
                    aj[c].coef = lrs[c]                     # per-chain learning rate
                ops.minibatch_fit(rows, gj, aj, E, T, self.mb_times, lrs[0], self.mb_cells, max_ctas)
                self.launches += 1
                return
            if len(set(lrs)) != 1:
                raise L.RcmarlError("the launch-chain mini-batch path takes one learning rate; use the persistent kernel")
            ops.minibatch_sgd(rows, gj, aj, E, T, self.mb_times, lrs[0], self.ws)
            self.launches += 2 * nb_steps
            return
        for e in range(E):
            for b in range(nb):
                cnt = min(self.mb_times, T - b * self.mb_times)
                rows.n_rows = cnt * N
                for c in range(nC):
                    gj[c].time_idx = base + 4 * ((c * E + e) * T + b * self.mb_times)
                    aj[c].coef = lrs[c] * 2.0 / (cnt * N * self.world)
                    if e == 1 and b == 0:
                        aj[c].loss_out = None                              # history['loss'][0]: epoch 0 only
                ops.grad(rows, gj, L.LOSS_MSE, self.ws)
                self._allreduce(self.sums_mb[:nC])
                ops.sgd_apply(aj)
                self.launches += 3

    def _minibatch_adam(self, adv, T, Ta, a0):
        """actor.fit(batch_size=200, epochs=1) of the adversaries (adversarial:41,116,224)."""
        N = self.N
        perms = torch.stack([self._perm(Ta) for _ in adv]).to(self.dev)    # [A, Ta], indices inside the actor window
        self.h2d_bytes += 4 * perms.numel()
        base = perms.data_ptr()
        nb = (Ta + self.actor_mb_times - 1) // self.actor_mb_times
        rows = self._rows(a0, 0, perms)
        gj = []
        for n, i in enumerate(adv):
            gj.append(ops.grad_job(self.actor[i], self.delta[i], self.sums_actor[n], L.IN_S, action_agent=i, time_idx=perms))
            self.loss_a[i:i + 1].zero_()
        gj = (L.GradJob * len(gj))(*gj)
        for b in range(nb):
            cnt = min(self.actor_mb_times, Ta - b * self.actor_mb_times)
            rows.n_rows = cnt * N
            aj = []
            for n, i in enumerate(adv):
                gj[n].time_idx = base + 4 * (n * Ta + b * self.actor_mb_times)
                self.adam_t[i] += 1
                aj.append(ops.adam_job(self.actor[i], self.adam_m[i], self.adam_v[i], self.sums_actor[n], self.PA,
                                       1.0 / (cnt * N * self.world), ops.keras_adam_lr_t(self.slow_lr[i], self.adam_t[i]),
                                       loss_out=self.loss_a[i:i + 1], loss_coef=1.0 / (Ta * N * self.world), loss_accumulate=1))
            ops.grad(rows, gj, L.LOSS_CE, self.ws)
            self._allreduce(self.sums_actor[:len(adv)])
            ops.adam_apply(aj)
            self.launches += 3

    # ------------------------------------------------------------------ checkpoint / resume
    def state_dict(self, include_buffer=True):
        """Everything needed to continue training bit-for-bit: parameters, Keras-Adam slots and step counts, the
        replay buffer, the episode counter that keys the Philox streams and the shuffle generator.  (The reference
        saves only the final weights, main.py:119-121; optimiser state and buffer are lost there -- SURVEY 5.)"""
        T = self.t_filled * self.N
        sd = dict(version=1, labels=list(self.labels), n_envs=self.N, t_filled=self.t_filled,
                  episodes_done=self.episodes_done, adam_t=list(self.adam_t), perm_rng=self._perm_gen.get_state(),
                  actor=self.actor.cpu(), critic=self.critic.cpu(), tr=self.tr.cpu(), critic_local=self.critic_local.cpu(),
                  adam_m=self.adam_m.cpu(), adam_v=self.adam_v.cpu())
        if include_buffer:
            sd.update(sa=self.sa[:T].cpu(), ns=self.ns[:T].cpu(), r=self.r[:T].cpu())
        return sd

    def load_state_dict(self, sd):
        if list(sd["labels"]) != list(self.labels) or int(sd["n_envs"]) != self.N:
            raise L.RcmarlError("checkpoint was written for a different agent set / environment count")
        for name in ("actor", "critic", "tr", "critic_local", "adam_m", "adam_v"):
            getattr(self, name).copy_(sd[name])
        self.adam_t = [int(t) for t in sd["adam_t"]]
        self.episodes_done = int(sd["episodes_done"])
        self._perm_gen.set_state(sd["perm_rng"])
        self.t_filled = 0
        if "sa" in sd:
            T = int(sd["t_filled"]) * self.N
            if T > self.sa.shape[0]:
                raise L.RcmarlError("checkpointed replay buffer does not fit")
            self.sa[:T].copy_(sd["sa"]); self.ns[:T].copy_(sd["ns"]); self.r[:T].copy_(sd["r"])
            self.t_filled = int(sd["t_filled"])

    def save(self, path, include_buffer=True):
        torch.save(self.state_dict(include_buffer), path)

    def load(self, path):
        self.load_state_dict(torch.load(path, map_location="cpu", weights_only=True))

    def trim(self):
        """Keep the newest `buffer_size` time rows (train_agents.py:158-163): chunked, non-overlapping
        device-to-device copies (pure data movement)."""
        q = self.t_filled - self.buffer_size
        if q <= 0:
            return
        N = self.N
        keep = self.buffer_size
        for buf in (self.sa, self.ns, self.r):
            done = 0
            while done < keep:
                n = min(q, keep - done)
                buf[done * N:(done + n) * N].copy_(buf[(done + q) * N:(done + q + n) * N])
                done += n
        self.t_filled = keep
