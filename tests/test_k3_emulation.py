"""K3's sampling arithmetic on the host (tests/k3emul.py), over every one of the 2^24 uniforms the kernel can
draw: the threshold without the clamp at 0 picks masked actions, the clamped one never does, and the clamped
one is the float64 inverse CDF except within the float32 rounding band of a bin edge."""
import numpy as np

import k3emul as K
from bbgpu import philox

F = np.float32


def _rows():
    """Random rows (30 % valid, logit scales 0.5 to 8) of which the first, fourth and sixth let the unclamped
    threshold pick a masked action (actions 12, 12 and 4), and one constructed row: tiny mass in lane 0,
    the heavy lane 1 with its first action masked."""
    rs = np.random.RandomState(0)
    rows = []
    for trial in range(6):
        valid = rs.rand(192) < 0.3
        valid[rs.randint(192)] = True
        z = (rs.randn(192) * rs.choice([0.5, 2, 4, 8])).astype(F)
        if trial in (0, 3, 5):
            rows.append((K.exp_terms(z, valid), valid))
    valid = np.zeros(192, bool)
    valid[[0, 1, 20, 21]] = True                     # lane 0: actions 0, 1; lane 1: 20, 21 (4 is masked)
    e = np.zeros(192, F)
    e[0], e[1], e[20], e[21] = 2.0 ** -23, 2.0 ** -24, 1.0, 0.5
    rows.append((e, valid))
    return rows


def test_unclamped_threshold_picks_masked_actions_and_the_clamp_stops_it():
    bad_old = []
    for e, valid in _rows():
        old = K.pick(e, valid, fixed=False)
        new = K.pick(e, valid, fixed=True)
        bad_old.append(int((~valid[old]).sum()))
        assert valid[new].all()
        # the clamp only changes draws where the old threshold was negative (t in the rounding gap)
        diff = old != new
        assert (~valid[old[diff]]).all()
    assert all(b > 0 for b in bad_old), bad_old


def test_clamped_pick_is_the_float64_inverse_cdf_outside_the_rounding_band():
    """Float64 reference: u * S over the exact prefix sums of the same e in sample_order().  The kernel's
    comparison t <= CDF_j involves at most 48 rounded additions in the lane, 2 in the scan, the exclusive
    prefix's subtraction, u * S and the 2 additions of S: 54 roundings of at most half an ulp of S each,
    so a draw may land in a neighbouring bin only within 27 ulp(S) of the edge between them."""
    order = philox.sample_order()
    for e, valid in _rows():
        got = K.pick(e, valid)
        e64 = e[order].astype(np.float64)
        hi = np.cumsum(e64)
        lo = hi - e64
        S = hi[-1]
        band = 27 * float(np.spacing(F(S)))
        x = K.ALL_U.astype(np.float64) * S
        ref = order[np.minimum(np.searchsorted(hi, x, side="right"), 191)]
        pos = K.sample_position()[got]
        inside = (x >= lo[pos] - band) & (x < hi[pos] + band)
        off = got != ref
        assert inside.all(), (np.flatnonzero(~inside)[:5], got[~inside][:5], ref[~inside][:5])
        assert valid[got].all() and (e[got] > 0).all()
        # what the band allows is rare: the draws it covers are a small share of all 2^24
        assert off.sum() <= (2 * band / S * 2 ** 24 + 1) * int((e > 0).sum()), off.sum()


def test_emulator_order_is_philox_sample_order():
    assert np.array_equal(K.ACTS.reshape(-1), philox.sample_order())
    assert np.array_equal(K.sample_position()[philox.sample_order()], np.arange(192))
