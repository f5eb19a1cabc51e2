"""The first pass of a batch larger than one wave of CTAs runs its last rounds over the packed unfinished problems
(mpcb_solve_cls_kernel, then one mpcb_solve_round_kernel per further round).  Each problem's arithmetic is the same as
when all its rounds run in the class kernel, which is what a batch of at most one wave does: the compacted solve of a
large batch must equal, bit for bit, the same problems solved in parts of one wave each."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SOLVE_THREADS, SOLVE_CTAS = 128, 2          # problems per CTA and CTAs per SM of the first pass (mpcb_api.cu)
CLS_ROUNDS = 4                              # rounds the class kernel runs before compacting


@pytest.mark.parametrize("caps", [dict(),
                                  dict(thread_max_rounds=6, thread_max_segments=4, thread_fail_rounds=0),
                                  dict(thread_max_rounds=4, thread_max_segments=2, thread_fail_rounds=0),
                                  dict(thread_max_segments=3)],
                         ids=["default", "rounds6", "rounds4", "fleet"])
def test_compacted_first_pass_is_bitwise_equal(caps, gpu_trackers, port_tables):
    import torch
    import safe_autonomous_driving_mpc_b200 as M
    from oracle import tracker_port as P
    L, _ = gpu_trackers[3]
    T = M.BatchedTracker(L, **caps)
    wave = torch.cuda.get_device_properties(0).multi_processor_count * SOLVE_CTAS * SOLVE_THREADS
    B = 65536
    assert B > wave, "the batch must be more than one wave of CTAs to be compacted"
    x0, obs, n = P.monte_carlo_problems(port_tables[3], B)
    dev = torch.device("cuda:0")
    d = [torch.from_numpy(a).to(dev) for a in (x0, obs, n)]
    n0 = T.launch_count()
    full = T.solve_batch(*d)
    torch.cuda.synchronize()
    launches_full = T.launch_count() - n0
    full = {k: v.cpu().numpy() for k, v in full.items()}
    parts = []
    n0 = T.launch_count()
    for lo in range(0, B, wave):
        r = T.solve_batch(*(a[lo:lo + wave].contiguous() for a in d))
        torch.cuda.synchronize()
        parts.append({k: v.cpu().numpy() for k, v in r.items()})
    launches_part = (T.launch_count() - n0) // len(parts)
    # the full batch ran one round kernel per round after the class kernel's, the parts none
    max_rounds = min(caps.get("thread_max_rounds", 5), 6)
    assert launches_full - launches_part == max(0, max_rounds - CLS_ROUNDS)
    for k in full:
        got = np.concatenate([p[k] for p in parts])
        assert np.array_equal(full[k], got, equal_nan=True), k
    assert (full["status"] == 0).mean() > 0.9
