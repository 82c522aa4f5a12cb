"""Host emulation, in float32 numpy, of the sampling arithmetic of K3 (bb_masked_sample_kernel, MODE 0) for
one row, in the kernel's order of operations:

- lane l of the 4-lane row group holds register i = 4k + c = action 16k + 4l + c;
- each lane keeps the running sum of its 48 terms e (its local CDF) and its total;
- S is the xor-1 / xor-2 butterfly of the lane totals, t = u * S;
- the lane's inclusive prefix comes from a Hillis-Steele scan (shfl_up by 1, then by 2);
- the owner lane L is the first lane with prefix > t and mass > 0 (``hit`` ballot), else the last lane
  with mass (``nz`` ballot);
- the local threshold is tl = t - (incl - tot), the pick is min(#{CDF entries <= tl}, last valid register).

The per-action terms e are an input, so the question of how exact ``ex2.approx`` is stays outside: feed
it e values that are exact (powers of two) to replay the device bit for bit, or ``exp_terms`` for a
float32 stand-in.  ``fixed=False`` is the threshold without the clamp at 0 (before it was added), which
can pick a masked action."""
import numpy as np

F = np.float32
LOG2E = F(1.4426950408889634)
# ACTS[l, i]: the action in register i of lane l
ACTS = np.array([[16 * (i >> 2) + 4 * l + (i & 3) for i in range(48)] for l in range(4)], dtype=np.int64)
ALL_U = np.arange(2 ** 24, dtype=np.float32) * F(2.0 ** -24)      # every uniform the kernel can draw


def exp_terms(z, valid):
    """float32 e[192] the way the kernel forms them, with np.exp2 standing in for ex2.approx:
    d2 = fma(z, log2e, -m * log2e) (the float64 product of two floats is exact, so one rounding),
    e = 2^d2, and e = 0 where masked."""
    z = np.asarray(z, F)
    valid = np.asarray(valid, bool)
    if not valid.any():
        return np.zeros(192, F)
    m = z[valid].max()
    nm2 = F(-m * LOG2E)
    d2 = (z.astype(np.float64) * float(LOG2E) + float(nm2)).astype(F)
    return np.where(valid, np.exp2(d2), F(0)).astype(F)


def pick(e, valid, u=ALL_U, fixed=True):
    """int64 actions the kernel draws for the uniforms u (float32, multiples of 2^-24) on the row whose
    per-action terms are e (float32[192], 0 where masked) and whose mask is valid (bool[192])."""
    e = np.asarray(e, F)
    valid = np.asarray(valid, bool)
    u = np.asarray(u, F)
    if not valid.any():
        return np.zeros(u.shape, np.int64)
    el = e[ACTS]                                      # [4, 48]
    cdf = np.zeros((4, 48), F)
    for l in range(4):
        run = F(0)
        for i in range(48):
            run = F(run + el[l, i])
            cdf[l, i] = run
    tot = cdf[:, -1].copy()
    b1 = [F(tot[l] + tot[l ^ 1]) for l in range(4)]                  # xor-1 butterfly
    s = F(b1[0] + b1[2])                                              # xor-2: the same value in every lane
    inc1 = [tot[0]] + [F(tot[l] + tot[l - 1]) for l in range(1, 4)]  # Hillis-Steele, d = 1
    incl = inc1[:2] + [F(inc1[l] + inc1[l - 2]) for l in range(2, 4)]  # d = 2
    t = (u * s).astype(F)
    hit = np.full(t.shape, -1, np.int64)
    for l in reversed(range(4)):
        hit = np.where((incl[l] > t) & (tot[l] > 0), l, hit)
    nz = [l for l in range(4) if tot[l] > 0]
    L = np.where(hit >= 0, hit, nz[-1] if nz else 0)
    excl = np.array([F(incl[l] - tot[l]) for l in range(4)], F)
    tl = (t - excl[L]).astype(F)
    if fixed:
        tl = np.maximum(tl, F(0))
    act = np.empty(t.shape, np.int64)
    for l in range(4):
        sel = L == l
        cnt = np.searchsorted(cdf[l], tl[sel], side="right")        # the CDF is non-decreasing
        v = np.nonzero(valid[ACTS[l]])[0]
        last = int(v[-1]) if v.size else 0
        act[sel] = ACTS[l][np.minimum(cnt, last)]
    return act


def sample_position():
    """int64 [192]: position of each action in the kernel's CDF order (inverse of philox.sample_order())."""
    pos = np.empty(192, np.int64)
    pos[ACTS.reshape(-1)] = np.arange(192)
    return pos
