"""The one-segment first pass (the default caps) keeps its factor and lane sensitivities in tensor memory: every CTA of
mpcb_solve_cls_kernel / mpcb_solve_round_kernel allocates 256 columns, so CTAs of batches in flight on other streams
share an SM's tensor memory.  A problem's answer must not depend on what else runs: each batch solved concurrently with
others must equal, bit for bit, the same batch solved alone.  Ragged sizes leave a partly filled CTA in every class,
whose empty lanes run each round with their warp; a multi-segment cap runs the instantiations without tensor memory."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SIZES = (65535, 24001, 65536)


def _problems(port_tables, i, B, seed):
    from oracle import tracker_port as P
    x0, obs, n = P.monte_carlo_problems(port_tables[i], B)
    perm = np.random.default_rng(seed).permutation(B)
    return x0[perm].copy(), obs[perm].copy(), n[perm].astype(np.int32)


def _bytes(out):
    return {k: v.cpu().numpy().tobytes() for k, v in out.items()}


@pytest.mark.parametrize("caps", [dict(), dict(thread_max_segments=3)], ids=["one_segment", "three_segments"])
@pytest.mark.parametrize("in_flight", [2, 3])
def test_batches_in_flight_equal_batches_alone(caps, in_flight, gpu_trackers, port_tables):
    import torch
    import safe_autonomous_driving_mpc_b200 as M
    dev = torch.device("cuda:0")
    routed = M.BatchedTracker([gpu_trackers[i][0] for i in (1, 2, 3)], **caps)
    jobs = []   # (tracker, device inputs, route)
    for c in range(in_flight):
        B = SIZES[c]
        if c == 2:   # a routed call: problems of all three routes in one batch
            x0, obs, n = _problems(port_tables, 3, B, seed=c)
            route = torch.from_numpy(np.random.default_rng(7).integers(0, 3, B).astype(np.int32)).to(dev)
            T = routed
        else:
            x0, obs, n = _problems(port_tables, c + 1, B, seed=c)
            route = None
            T = M.BatchedTracker(gpu_trackers[c + 1][0], **caps)
        jobs.append((T, [torch.from_numpy(a).to(dev) for a in (x0, obs, n)], route))
    alone = []
    for T, d, route in jobs:
        r = T.solve_batch(*d, route=route)
        torch.cuda.synchronize()
        alone.append(_bytes(r))
    streams = [torch.cuda.Stream(dev) for _ in jobs]
    for rep in range(2):
        outs = [T.solve_batch(*d, stream=s.cuda_stream, route=route) for (T, d, route), s in zip(jobs, streams)]
        torch.cuda.synchronize()
        for c, (o, a) in enumerate(zip(outs, alone)):
            got = _bytes(o)
            for k in a:
                assert got[k] == a[k], f"batch {c} ({SIZES[c]} problems), output {k}, repetition {rep}"
