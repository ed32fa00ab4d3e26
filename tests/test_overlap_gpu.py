"""The C2 update round with the adversaries' mini-batch chains on a second stream beside the cooperative full-batch fits
(rcmarl_overlap_split): reproducible bit for bit from run to run, and the two phases really run at the same time."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


def need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


def c2_trainer():
    import bench
    from rcmarl.trainer import Trainer
    cfg = bench.workload("C2", 4096)
    tr = Trainer(seed=1, **cfg)
    tr.rollout_block()
    tr.rollout_block()
    return tr


def test_two_overlapped_c2_rounds_are_bitwise_reproducible():
    need_gpu()
    runs = []
    for _ in range(2):
        tr = c2_trainer()
        losses = [tr.update_round()]
        assert tr._side is not None, "the C2 round should overlap the chains with the fits"
        tr.rollout_block()
        losses.append(tr.update_round())
        torch.cuda.synchronize()
        runs.append(([x.cpu().numpy().copy() for x in (tr.actor, tr.critic, tr.tr, tr.critic_local)], losses))
    (pa, la), (pb, lb) = runs
    for a, b in zip(pa, pb):
        assert np.array_equal(a, b)
    for x, y in zip(la, lb):
        for k in x:
            assert np.array_equal(x[k], y[k]), k


def test_chains_and_fits_run_at_the_same_time():
    need_gpu()
    from torch.profiler import ProfilerActivity, profile
    tr = c2_trainer()
    tr.update_round()                                   # warm up
    tr.rollout_block()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        tr.update_round()
        torch.cuda.synchronize()
    kern = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    mb = [(e.time_range.start, e.time_range.end) for e in kern if "mb_persist_ws_kernel" in e.name]
    fit = [(e.time_range.start, e.time_range.end) for e in kern if "grad_kernel_ws" in e.name]
    assert len(mb) == tr.n_epochs and len(fit) >= 5 * tr.n_epochs
    both = sum(max(0.0, min(e, e0) - max(s, s0)) for s, e in fit for s0, e0 in mb)
    alone = sum(e - s for s, e in fit)
    # most of the full-batch fits' kernel time lies inside the chains' kernels
    assert both > 0.5 * alone, (both, alone)
