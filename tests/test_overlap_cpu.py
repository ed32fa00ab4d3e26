"""Host arithmetic of rcmarl_overlap_split (no device): how an update round splits the SMs between the cooperative
full-batch fits and the adversaries' mini-batch chains when both run at the same time, and when it stays serial."""
import numpy as np

from rcmarl import _lib as L
from rcmarl import ops

SA, S = L.IN_SA, L.IN_S
C2 = dict(n_agents=5, fit_kinds=[SA, S] * 4, fit_rows=3000 * 4096, fit_launches=5, chain_kinds=[S, SA, S],
          mb_rows=32 * 4096, mb_steps=940, world=1, sm_count=148)


def split(**kw):
    return ops.overlap_split(**{**C2, **kw})


def chain_shares(budget, mb_rows=C2["mb_rows"], kinds=C2["chain_kinds"]):
    import ctypes as C
    k = (C.c_int32 * len(kinds))(*kinds)
    out = (C.c_int32 * len(kinds))()
    L.check(L.lib().rcmarl_grad_grid_plan(5, k, len(kinds), L.LOSS_MSE, mb_rows, 1, budget, out), "rcmarl_grad_grid_plan")
    return list(out)


def test_c2_splits_the_gpu_between_fits_and_chains():
    fit, chains = split()
    assert fit + chains == 148
    assert fit % 8 == 0 and fit >= 8 and chains >= 3
    assert (fit, chains) == (72, 76)
    assert chain_shares(chains) == [25, 26, 25]              # cost-sized shares inside the chains' budget


def test_serial_when_there_is_nothing_to_overlap_or_ranks_must_agree():
    assert split(chain_kinds=[]) is None                    # C1 / C3: all-cooperative teams
    assert split(fit_kinds=[]) is None                      # no cooperative agent
    assert split(world=2) is None and split(world=8) is None
    assert split(n_agents=16) is None                       # the 16-agent kernels have no measured cost model
    assert split(mb_steps=0) is None and split(fit_launches=0) is None
    assert split(sm_count=10) is None                       # fewer SMs than jobs + chains


def test_serial_when_the_model_predicts_no_gain():
    # a few thousand buffer rows: both phases are fixed cost, nothing to gain from fewer SMs each
    assert split(fit_rows=32 * 64, mb_rows=64) is None


def test_budgets_hold_for_any_mix():
    rs = np.random.RandomState(0)
    for _ in range(300):
        nf, nc = int(rs.randint(1, 17)), int(rs.randint(1, 7))
        sms = int(rs.randint(1, 200))
        kw = dict(fit_kinds=[int(v) for v in rs.randint(0, 2, nf)], chain_kinds=[int(v) for v in rs.randint(0, 2, nc)],
                  fit_rows=int(rs.randint(1, 1 << 25)), mb_rows=int(rs.randint(1, 1 << 18)),
                  fit_launches=int(rs.randint(1, 8)), mb_steps=int(rs.randint(1, 3000)), sm_count=sms)
        got = split(**kw)
        if got is None:
            continue
        fit, chains = got
        assert fit + chains <= sms
        assert fit >= nf and fit % nf == 0 and chains >= nc
