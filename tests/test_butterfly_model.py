"""CPU model of the butterfly ("transpose") warp reduction of the per-Gaussian backward
(gsplat_b200/csrc/common.cuh: Butterfly<M,16> + butterfly_slot<M>; pergauss.cu uses M = 12 for the pose
gradient and M = 3 for the view-direction sum).  The recursion is restated in numpy with an explicit
shfl_xor so that slot ownership and sums can be checked; the template is generic in M, so a spread of
M is checked, including M > 32."""
import numpy as np
import pytest


def butterfly(vals):
    """vals: [32, M] per-lane values -> per-lane v[0] after the reduction."""
    v = vals.astype(np.float64).copy()
    lanes = np.arange(32)
    m = v.shape[1]
    for off in (16, 8, 4, 2, 1):
        if m > 1:
            h = (m + 1) // 2
            up = (lanes & off) != 0
            new = np.zeros((32, h))
            for i in range(h):
                hi = v[:, i + h] if i + h < m else np.zeros(32)
                send = np.where(up, v[:, i], hi)
                keep = np.where(up, hi, v[:, i])
                new[:, i] = keep + send[lanes ^ off]
            v, m = new, h
        else:
            v = v + v[lanes ^ off]
    return v[:, 0]


def slot_of(lane, M):
    mt, mr, slot, primary = M, M, 0, True
    for off in (16, 8, 4, 2, 1):
        if mt > 1:
            h = (mt + 1) // 2
            if lane & off:
                slot += h
                mr = mr - h if mr > h else 0
            else:
                mr = min(mr, h)
            mt = h
        elif lane & off:
            primary = False
    return slot if (mr >= 1 and primary) else -1


@pytest.mark.parametrize("M", [7, 8, 9, 10, 11, 12, 13, 14, 16, 22, 24, 38, 40])
def test_every_slot_owned_once_with_the_right_sum(M):
    rng = np.random.RandomState(M)
    vals = rng.standard_normal((32, M))
    out = butterfly(vals)
    owners = {}
    for lane in range(32):
        s = slot_of(lane, M)
        if s >= 0:
            assert s < M and s not in owners, f"slot {s} owned twice"
            owners[s] = lane
    if M <= 32:
        assert sorted(owners) == list(range(M)), f"unowned slots for M={M}"
    for s, lane in owners.items():
        assert abs(out[lane] - vals[:, s].sum()) < 1e-9
