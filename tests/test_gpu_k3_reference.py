"""K3 (bb_masked_sample, all three modes) and the policy-head backward / fused PPO loss against float64 references,
at rollout and minibatch sizes that run the persistent kernels for one and for many trips, on random rows
and on edge rows.  u = 2^-24 below; K3 forms e_i = ex2.approx(fma(z_i, log2e, -m log2e)) (relative error
2^-22 = 4u), sums 48 terms per lane and then across 4 lanes in float32.  The bounds used by the tests:

- S (and every CDF entry relative to S): at most 54 roundings of half an ulp (48 in the lane, 2 in the scan,
  the exclusive prefix, 2 for S, u * S), 4u from ex2.approx, and the rounding of each exponent argument,
  |d_i| u relative for term i, i.e. A u S in total with A = sum_i q_i |d_i| (q the probabilities, d in
  nats).  The rounding of -m log2e is common to all terms and cancels.  Band: u S (64 + 2A).
- log p_a = d_a - log S: u (4 (|m| + |d_a| + |log S|) + 64).
- entropy log S - sum q_i d_i: u (64 (1 + A) + 4 |log S|); network.py's clamp of q at 1e-10 moves the
  reference by less than 192 * 1e-10 * 23 < 8u, inside the constant.
"""
import math

import numpy as np
import pytest

import k3emul as K

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
EPS = float(np.finfo(np.float32).eps)
LOG_EPS = float(np.float32(math.log(EPS)))
LOG_1M_EPS = float(np.float32(math.log1p(-EPS)))
GUARD = 64
SIZES = [4096, 23679, 23681, 28417, 94723, 262144, 1048573]
CHUNK = 1 << 16


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


def _planes(torch, valid):
    from bbgpu.network import _pack_mask_planes
    return _pack_mask_planes(valid).contiguous()


def _edge_rows():
    """float32 logits and bool masks of the edge rows, [E, 192] each."""
    rs = np.random.RandomState(21)
    zs, vs = [], []

    def add(z, v):
        zs.append(np.asarray(z, np.float32))
        vs.append(np.asarray(v, bool))

    def base():
        return (rs.randn(192) * 2).astype(np.float32)

    add(base(), np.zeros(192, bool))                                   # all masked
    for l in range(4):                                                 # one valid action, every lane and c
        for c in range(4):
            v = np.zeros(192, bool)
            v[16 * ((4 * l + c) % 12) + 4 * l + c] = True
            add(base(), v)
    v = np.zeros(192, bool)
    v[[176 + 4 * l + 3 for l in range(4)]] = True                      # only the last action of each lane
    add(base(), v)
    for l in range(4):
        v = np.zeros(192, bool)
        v[176 + 4 * l + 3] = True
        v[rs.randint(0, 176)] = True
        add(base(), v)
    for top in (0, 95, 191):                                           # the rest 100 to 300 below the maximum
        z = base()
        v = rs.rand(192) < 0.5
        v[top] = True
        z[v] = np.float32(3.0) - np.float32(100) - (rs.rand(int(v.sum())) * 200).astype(np.float32)
        z[top] = 3.0
        add(z, v)
    z = np.full(192, -1.0, np.float32)                                 # exact ties within and across lanes
    z[[4, 5, 6, 20, 36, 100, 191]] = 2.5
    add(z, np.ones(192, bool))
    add((rs.randint(-3, 3, 192) * 0.5).astype(np.float32), rs.rand(192) < 0.7)
    for mag in (0.01, 1.0, 3.0, -7.0, 30.0):                           # near-ties 1 to 3 ulps apart
        for k in (1, 2, 3):
            z = (np.float32(mag) - np.float32(abs(mag) + 1) * rs.rand(192).astype(np.float32)).astype(np.float32)
            v = rs.rand(192) < 0.7
            hi = np.float32(mag)
            for _ in range(k):
                hi = np.nextafter(hi, np.float32(np.inf))
            lo_pos, hi_pos = sorted(rs.choice(192, 2, replace=False))
            z[lo_pos], z[hi_pos] = np.float32(mag), hi             # the larger logit at the higher index
            v[[lo_pos, hi_pos]] = True
            add(z, v)
            z2 = z.copy()
            z2[lo_pos], z2[hi_pos] = hi, np.float32(mag)            # and at the lower index
            add(z2, v)
    return np.stack(zs), np.stack(vs)


def _rows(torch, n, seed):
    """Random rows (logit scale 0.5 to 8, 1 to 100 % valid, at least one valid action) with the edge rows
    at the start and at the end of the batch (the tail runs on the last trip of the persistent warps)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    z = torch.randn(n, 192, device="cuda", generator=g) * (0.5 * 16 ** torch.rand(n, 1, device="cuda", generator=g))
    valid = torch.rand(n, 192, device="cuda", generator=g) < 0.01 + 0.99 * torch.rand(n, 1, device="cuda", generator=g)
    valid[torch.arange(n, device="cuda"), torch.randint(0, 192, (n,), device="cuda", generator=g)] = True
    ez, ev = _edge_rows()
    E = ez.shape[0]
    z[:E], valid[:E] = torch.from_numpy(ez).cuda(), torch.from_numpy(ev).cuda()
    z[n - E:], valid[n - E:] = torch.from_numpy(ez).cuda(), torch.from_numpy(ev).cuda()
    return z, valid


def _ref(torch, z64, valid):
    """float64 terms of the masked categorical head: d = z - m (-inf where masked), e = exp(d), S, log S,
    entropy (network.py's formula) and A = sum q |d|."""
    anyv = valid.any(1)
    zm = z64.masked_fill(~valid, float("-inf"))
    m = torch.where(anyv, zm.max(1).values, torch.zeros_like(zm[:, 0]))
    d = zm - m[:, None]
    e = torch.exp(d)
    S = e.sum(1)
    logS = torch.log(S)
    q = e / S[:, None].clamp(min=1e-10)
    dq = torch.where(valid, d, torch.zeros_like(d))
    H = -(q * torch.log(q.clamp(min=1e-10)) * valid).sum(1)
    A = (q * dq.abs()).sum(1)
    return dict(m=m, d=d, e=e, S=S, logS=logS, H=torch.where(anyv, H, torch.zeros_like(H)), A=A, any=anyv)


def _logp_ref(torch, r, act, valid):
    """float64 log p of the given actions with Categorical's clamp; log eps for masked / out-of-range
    actions, log(1 - eps) on all-masked rows (what the kernel defines there)."""
    inr = (act >= 0) & (act < 192)
    a = torch.where(inr, act, torch.zeros_like(act)).long()
    ok = inr & valid.gather(1, a[:, None])[:, 0]
    da = r["d"].gather(1, a[:, None])[:, 0]
    lp = torch.where(ok, da - r["logS"], torch.full_like(da, LOG_EPS)).clamp(LOG_EPS, LOG_1M_EPS)
    lp = torch.where(r["any"], lp, torch.full_like(lp, LOG_1M_EPS))
    tol = U * (4 * (r["m"].abs() + torch.where(ok, da.abs(), torch.zeros_like(da)) + r["logS"].abs()) + 64)
    return lp, torch.where(r["any"], tol, torch.full_like(tol, U)), da


def _outs(torch, n):
    act = torch.full((n + GUARD,), -7, dtype=torch.int32, device="cuda")
    lp = torch.full((n + GUARD,), 123.0, device="cuda")
    en = torch.full((n + GUARD,), 456.0, device="cuda")
    return act, lp, en


def _guards_intact(torch, act, lp, en, n):
    assert (act[n:] == -7).all() and (lp[n:] == 123.0).all() and (en[n:] == 456.0).all(), "wrote past row n"


# ------------------------------------------------------------------------------------------------- a
def _sweep_patterns():
    """16 rows: 12 generic random rows (30 % valid, scales 0.5 to 8) and 4 built to hit the rounding gap of
    the exclusive prefix: lane 0 holds r ulp(1) of mass (r in (0.5, 1): 1 + a0 rounds up), the heavy lane L
    holds the maximum (e = 1) at action 16 + 4L with its first action 4L masked, and a third lane holds
    mass r, which puts S near 1 + r and the draw u = 2^-24 inside the gap."""
    rs = np.random.RandomState(0)
    zs, vs = [], []
    for _ in range(12):
        v = rs.rand(192) < 0.3
        v[rs.randint(192)] = True
        zs.append((rs.randn(192) * rs.choice([0.5, 2, 4, 8])).astype(np.float32))
        vs.append(v)
    for L, other, r in ((1, 3, 0.7), (2, 1, 0.6), (3, 2, 0.8), (1, 2, 0.75)):
        z = np.full(192, -50.0, np.float32)
        v = np.zeros(192, bool)
        z[0], v[0] = math.log(r * 2.0 ** -23), True
        z[16 + 4 * L], v[16 + 4 * L] = 0.0, True
        z[16 * 5 + 4 * other + 1], v[16 * 5 + 4 * other + 1] = math.log(r), True
        v[rs.rand(192) < 0.1] = True                             # a few more valid actions far below (e ~ 2e-22)
        v[4 * L] = False
        zs.append(z)
        vs.append(v)
    return np.stack(zs), np.stack(vs)


@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
def test_sampling_never_picks_a_masked_action(torch, dtype):
    """2^20 rows (16 patterns tiled) x 256 call counters = 2^28 draws: every sampled action must be valid."""
    from bbgpu import capi
    pz, pv = _sweep_patterns()
    n = 1 << 20
    logits = torch.from_numpy(pz).cuda().repeat(n // 16, 1).to(getattr(torch, dtype)).contiguous()
    pvalid = torch.from_numpy(pv).cuda()
    planes = _planes(torch, pvalid.repeat(n // 16, 1))
    pat = torch.arange(n, device="cuda") % 16
    act = torch.empty(n, dtype=torch.int32, device="cuda")
    bad = torch.zeros(16, dtype=torch.int64, device="cuda")
    for ctr in range(256):
        capi.masked_sample(logits, planes, n, 0x5EED, ctr, 0, act, None, None)
        ok = pvalid[pat, act.long()]
        bad += torch.bincount(pat[~ok], minlength=16)
    bad = bad.cpu().numpy()
    print("masked picks per pattern (%s):" % dtype, bad.tolist())
    assert bad.sum() == 0, "%d of 2^28 draws picked a masked action (per pattern: %s)" % (bad.sum(), bad.tolist())


# ------------------------------------------------------------------------------------------------- b
def _exact_logit(k):
    """float32 z with fl(z * log2e_f32) == -k, so that the kernel's exponent argument is exactly -k."""
    L = float(K.LOG2E)
    z = np.float32(-k / L)
    for _ in range(64):
        p = np.float32(float(z) * L)
        if p == -k:
            return z
        z = np.nextafter(z, np.float32(np.inf) if p < -k else np.float32(-np.inf))
    raise AssertionError("no float32 logit maps to exponent %d" % k)


def test_sampling_replays_the_emulator_on_an_exact_row(torch):
    """A row whose terms are exact powers of two (e = 2^-23, 2^-24 in lane 0, 1 and 1/2 in lane 1, action 4
    masked): every float32 sum of the kernel is then the emulator's.  1 + 1.5 * 2^-23 rounds up to
    1 + 2^-22, so the exclusive prefix of lane 1 exceeds the lane-0 mass and the draw u = 2 * 2^-24 falls
    in the gap; the (row, counter) whose Philox word gives that u is searched on the host.  The premise,
    that ex2.approx is exact at integer arguments, is checked on 2^20 ordinary draws of the same row."""
    from bbgpu import capi, philox
    z = np.full(192, -30.0, np.float32)
    valid = np.zeros(192, bool)
    for a, k in ((0, 23), (1, 24), (20, 0), (21, 1)):
        z[a], valid[a] = _exact_logit(k), True
    e = np.zeros(192, np.float32)
    e[[0, 1, 20, 21]] = [2.0 ** -23, 2.0 ** -24, 1.0, 0.5]
    table = K.pick(e, valid)                                     # fixed threshold, every u
    gap = np.flatnonzero(~valid[K.pick(e, valid, fixed=False)])  # u * 2^24 where the unclamped one fails
    assert gap.size > 0 and valid[table].all()
    seed, rows, ctrs = 1, 1 << 16, 256
    hit = None
    r = np.arange(rows, dtype=np.uint64)
    for c in range(ctrs):
        w = philox.philox4x32_10(r & philox.MASK32, r >> np.uint64(32), c, philox.STREAM_SAMPLE, seed, 0)[0] >> np.uint32(8)
        j = np.flatnonzero(np.isin(w, gap))
        if j.size:
            hit = (int(j[0]), c, int(w[j[0]]))
            break
    assert hit is not None, "no (row, counter) of the search space draws into the gap"
    row, ctr, uw = hit
    n = rows
    logits = torch.from_numpy(np.tile(z, (n, 1))).cuda()
    planes = _planes(torch, torch.from_numpy(np.tile(valid, (n, 1))).cuda())
    act, lp, en = _outs(torch, n)
    # premise: 16 counters x 65,536 rows = 2^20 ordinary draws equal the emulator bit for bit
    mism = 0
    for c in range(16):
        capi.masked_sample(logits, planes, n, seed, 1000 + c, 0, act[:n], lp[:n], en[:n])
        want = table[(philox.sample_uniforms(seed, 1000 + c, n) * np.float32(2 ** 24)).astype(np.int64)]
        mism += int((act[:n].cpu().numpy() != want).sum())
    assert mism == 0, ("ex2.approx is not exact at integer arguments on this device: %d of 2^20 draws differ "
                       "from the float32 emulation of the row" % mism)
    capi.masked_sample(logits, planes, n, seed, ctr, 0, act[:n], lp[:n], en[:n])
    _guards_intact(torch, act, lp, en, n)
    got = int(act[row])
    print("exact row: row %d counter %d u = %d * 2^-24 -> action %d (unclamped threshold: %d)"
          % (row, ctr, uw, got, int(K.pick(e, valid, np.array([uw * 2.0 ** -24], np.float32), fixed=False)[0])))
    assert valid[got] and got == int(table[uw])


# ------------------------------------------------------------------------------------------------- c, d
def _check_modes(torch, n, dtype, seed):
    from bbgpu import capi, philox
    dt = getattr(torch, dtype)
    z32, valid = _rows(torch, n, seed)
    logits = z32.to(dt).contiguous()
    del z32
    planes = _planes(torch, valid)
    order = torch.from_numpy(philox.sample_order()).cuda()
    pos_of = torch.from_numpy(K.sample_position()).cuda()
    row_offset, sseed, ctr = 977, 0xC0FFEE, 3
    u = torch.from_numpy(philox.sample_uniforms(sseed, ctr, row_offset + n)[row_offset:]).cuda().double()
    act, lp, en = _outs(torch, n)

    # MODE 0: sample
    capi.masked_sample(logits, planes, n, sseed, ctr, 0, act[:n], lp[:n], None, row_offset)
    _guards_intact(torch, act, lp, en, n)
    off = 0
    for c0 in range(0, n, CHUNK):
        c1 = min(n, c0 + CHUNK)
        v = valid[c0:c1]
        r = _ref(torch, logits[c0:c1].double(), v)
        a = act[c0:c1].long()
        anyv = r["any"]
        assert (a[~anyv] == 0).all()
        assert ((a >= 0) & (a < 192)).all()
        assert v.gather(1, a.clamp(0, 191)[:, None])[anyv, 0].all(), "sampled a masked action"
        eo = r["e"][:, order]
        hi = eo.cumsum(1)
        lo = hi - eo
        x = (u[c0:c1] * r["S"])[:, None]
        ref = order[torch.searchsorted(hi.contiguous(), x.contiguous(), right=True).clamp(max=191)[:, 0]]
        band = U * r["S"] * (64 + 2 * r["A"])
        p = pos_of[a][:, None]
        inside = (x[:, 0] >= lo.gather(1, p)[:, 0] - band) & (x[:, 0] < hi.gather(1, p)[:, 0] + band)
        bad = anyv & ~inside
        assert not bad.any(), ("sampled action outside its float64 bin + band", torch.nonzero(bad)[:5, 0] + c0)
        off += int((anyv & (a != ref)).sum())
        lp_ref, tol, _ = _logp_ref(torch, r, a.int(), v)
        err = (lp[c0:c1].double() - lp_ref).abs()
        assert (err <= tol).all(), ("log p of the sampled action", float((err / tol).max()))
    print("n=%d %s: %d of %d draws differ from the float64 inverse CDF, all inside the band" % (n, dtype, off, n))

    # MODE 1: argmax = float64 masked argmax, lowest index on ties
    capi.masked_sample(logits, planes, n, 0, 0, 1, act[:n], lp[:n], None)
    _guards_intact(torch, act, lp, en, n)
    for c0 in range(0, n, CHUNK):
        c1 = min(n, c0 + CHUNK)
        zm = logits[c0:c1].double().masked_fill(~valid[c0:c1], float("-inf"))
        mx = zm.max(1, keepdim=True).values
        first = torch.where(zm == mx, torch.arange(192, device="cuda"), torch.full_like(zm, 192, dtype=torch.long)).min(1).values
        want = torch.where(valid[c0:c1].any(1), first, torch.zeros_like(first))
        got = act[c0:c1].long()
        assert torch.equal(got, want), ("argmax", torch.nonzero(got != want)[:5, 0] + c0)

    # MODE 2: evaluate given actions, some of them masked or out of range
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    given = torch.multinomial(valid.float() + 1e-30 * (~valid.any(1, keepdim=True)).float(), 1, generator=g)[:, 0].int()
    k = torch.arange(n, device="cuda")
    masked_any = (~valid).any(1)
    first_masked = (~valid).int().argmax(1).int()
    sel = (k % 7 == 3) & masked_any
    given[sel] = first_masked[sel]
    given[k % 11 == 5] = -1
    given[k % 13 == 6] = 192
    given[k % 17 == 8] = 40000
    act[:n] = given
    capi.masked_sample(logits, planes, n, 0, 0, 2, act[:n], lp[:n], en[:n])
    _guards_intact(torch, act, lp, en, n)
    assert torch.equal(act[:n], given)
    for c0 in range(0, n, CHUNK):
        c1 = min(n, c0 + CHUNK)
        v = valid[c0:c1]
        r = _ref(torch, logits[c0:c1].double(), v)
        lp_ref, tol, _ = _logp_ref(torch, r, given[c0:c1], v)
        err = (lp[c0:c1].double() - lp_ref).abs()
        assert (err <= tol).all(), ("evaluate log p", float((err / tol).max()))
        tol_h = U * (64 * (1 + r["A"]) + 4 * r["logS"].abs())
        err_h = (en[c0:c1].double() - r["H"]).abs()
        assert (err_h <= tol_h).all(), ("entropy", float((err_h / tol_h).max()))
        assert (en[c0:c1][~r["any"]] == 0).all()


@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
@pytest.mark.parametrize("n", SIZES)
def test_sample_argmax_evaluate_match_float64(torch, n, dtype):
    """MODE 0 against the float64 inverse CDF over sample_order() with the stored Philox uniforms (nonzero
    row offset), MODE 1 against the float64 masked argmax, MODE 2 log p and entropy, at sizes on both sides
    of one resident wave (23,680 rows for float32, 28,416 for bfloat16) and up to 44 trips."""
    _check_modes(torch, n, dtype, seed=n % 1000 + (7 if dtype == "bfloat16" else 0))


# ------------------------------------------------------------------------------------------------- e
def _head64(torch, z, valid, act):
    """float64 log p (Categorical clamp) and entropy (network.py) of given valid actions, differentiable."""
    probs = torch.softmax(z.masked_fill(~valid, float("-inf")), -1)
    pn = probs / probs.sum(-1, keepdim=True)
    lp = torch.log(pn.clamp(EPS, 1 - EPS)).gather(1, act[:, None]).squeeze(1)
    q = probs / probs.sum(-1, keepdim=True).clamp(min=1e-10)
    return lp, -(q * torch.log(q.clamp(min=1e-10)) * valid).sum(-1), pn


def _grad_tol(torch, dtype, g1, g2, H, logS):
    """|dlogits - ref| <= rtol |ref| + atol_row.  p_i is good to (64 + 2 |d_i|) u relative, so 2^-16
    covers |d| up to ~90 (smaller p are below atol); the cancellations g1 (1 - p_a) and p_i (log p_i + H)
    leave an absolute error of the row's scale times that.  bfloat16 outputs add their rounding, 2^-9."""
    rtol = 2.0 ** -16 + (2.0 ** -8 if dtype == "bfloat16" else 0.0)
    return rtol, 2.0 ** -16 * (g1.abs() + g2.abs() * (1 + H.abs() + logS.abs()))


def _rows_close(got, ref, rtol, atol_row):
    err = (got.double() - ref).abs()
    return (err <= rtol * ref.abs() + atol_row[:, None]).all(1)


def _logp_grad64(torch, pn, act):
    """d log p_a / d z without Categorical's clamp: onehot(a) - p (0 on masked actions, where p = 0)."""
    gr = -pn
    return gr.scatter_add(1, act[:, None], torch.ones_like(pn[:, :1]))


def _check_grad(torch, got, ref_ent, g_lp, on, edge, rtol, atol, what):
    """got must equal ref_ent + [on] g_lp.  On an edge row (a decision within the kernel's rounding of its
    threshold) the other side, ref_ent + [not on] g_lp, is right as well.  Returns how many edge rows
    took the other side."""
    zero = torch.zeros_like(g_lp)
    ok = _rows_close(got, ref_ent + torch.where(on[:, None], g_lp, zero), rtol, atol)
    other = _rows_close(got, ref_ent + torch.where(on[:, None], zero, g_lp), rtol, atol)
    bad = ~ok & ~(edge & other)
    assert not bad.any(), (what, torch.nonzero(bad)[:5, 0].tolist())
    return int((~ok & edge).sum())


def _backward_inputs(torch, n, dtype, seed):
    z32, valid = _rows(torch, n, seed)
    anyv = valid.any(1)
    valid[~anyv, 0] = True                                   # the PPO update never sees an all-masked row
    g = torch.Generator(device="cuda").manual_seed(seed)
    act = torch.multinomial(valid.float(), 1, generator=g)[:, 0]
    return z32.to(getattr(torch, dtype)).contiguous(), valid, act, g


def _near_clamp(pa):
    """p_a within the kernel's error (2^-16 relative, see _grad_tol) of Categorical's clamp at eps or 1 - eps."""
    return ((pa - EPS).abs() < 2 ** -16 * EPS) | (((pa - (1 - EPS)).abs() < 2 ** -16) & (pa < 1))


@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
@pytest.mark.parametrize("n", [8192, 262144])
def test_masked_head_backward_matches_float64_autograd(torch, n, dtype):
    """bb_masked_head_backward against float64: autograd of network.py's entropy plus the closed form
    g_logp (onehot - p) of Categorical's log-prob where eps <= p_a <= 1 - eps.  A row whose p_a lies within
    the kernel's error of the clamp (p_a = 1 exactly is not such a row) may take either side."""
    from bbgpu import capi
    logits, valid, act, g = _backward_inputs(torch, n, dtype, seed=31 + n % 97)
    planes = _planes(torch, valid)
    g1 = torch.randn(n, device="cuda", generator=g)
    g2 = torch.randn(n, device="cuda", generator=g)
    out = torch.full((n + GUARD, 192), 77.0, device="cuda").to(logits.dtype)
    capi.masked_head_backward(logits, planes, n, act.int(), g1, g2, out[:n])
    torch.cuda.synchronize()
    assert (out[n:] == 77.0).all(), "wrote past row n"
    flipped = 0
    for c0 in range(0, n, CHUNK):
        c1 = min(n, c0 + CHUNK)
        v, a = valid[c0:c1], act[c0:c1]
        z = logits[c0:c1].double().requires_grad_(True)
        _, ent, pn = _head64(torch, z, v, a)
        (g2[c0:c1].double() * ent).sum().backward()
        with torch.no_grad():
            pa = pn.gather(1, a[:, None])[:, 0]
            on = (pa >= EPS) & (pa <= 1 - EPS)
            g_lp = g1[c0:c1].double()[:, None] * _logp_grad64(torch, pn, a)
            r = _ref(torch, logits[c0:c1].double(), v)
            rtol, atol = _grad_tol(torch, dtype, g1[c0:c1].double(), g2[c0:c1].double(), r["H"], r["logS"])
            flipped += _check_grad(torch, out[c0:c1], z.grad, g_lp, on, _near_clamp(pa), rtol, atol, "dlogits")
            assert (out[c0:c1][~v] == 0).all(), "nonzero gradient on a masked action"
    print("n=%d %s: %d rows at the clamp edge took the other side" % (n, dtype, flipped))


@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
@pytest.mark.parametrize("n", [8192, 262144])
def test_ppo_loss_matches_float64_autograd(torch, n, dtype):
    """bb_ppo_loss at the minibatch size (one trip) and at a rollout's 262,144 rows (22 trips of the capped
    grid, float partial sums per lane, one atomic set per warp), against float64: autograd of the entropy
    bonus plus the closed-form gradient of the clipped surrogate.  Rows within 2^-14 of a clip edge or near
    the log-prob clamp may take either side of that decision.  Sums: each row's term is within 2^-16 of
    its float64 value (relative, from log p's bound through exp), the per-lane float32 sums of up to 22
    rows and the 4-lane fold add < 2^-19: |sum - ref| <= 2^-15 sum |term| <= 2^-15 n max |term|.  The
    clip count may differ by the rows whose |r - 1| lies within 2^-14 of the clip (counted)."""
    from bbgpu import capi
    clip, vc, ec = 0.2, 0.5, 0.01
    logits, valid, act, g = _backward_inputs(torch, n, dtype, seed=57 + n % 89)
    planes = _planes(torch, valid)
    values = torch.randn(n, device="cuda", generator=g)
    ret = values + torch.randn(n, device="cuda", generator=g)
    adv = torch.randn(n, device="cuda", generator=g)
    with torch.no_grad():
        lp0 = torch.cat([_head64(torch, logits[c0:c0 + CHUNK].double(), valid[c0:c0 + CHUNK], act[c0:c0 + CHUNK])[0]
                         for c0 in range(0, n, CHUNK)])
    old = (lp0 + 0.25 * torch.randn(n, device="cuda", generator=g, dtype=torch.float64)).float()
    dl = torch.full((n + GUARD, 192), 77.0, device="cuda").to(logits.dtype)
    dv = torch.full((n + GUARD,), 77.0, device="cuda")
    sums = torch.zeros(5, dtype=torch.float64, device="cuda")
    capi.ppo_loss(logits, planes, n, act.int(), old, adv, ret, values, clip, vc, ec, dl[:n], dv[:n], sums)
    torch.cuda.synchronize()
    assert (dl[n:] == 77.0).all() and (dv[n:] == 77.0).all(), "wrote past row n"
    terms = torch.zeros(5, n, dtype=torch.float64, device="cuda")
    n_amb = 0
    flipped = 0
    for c0 in range(0, n, CHUNK):
        c1 = min(n, c0 + CHUNK)
        v, a = valid[c0:c1], act[c0:c1]
        z = logits[c0:c1].double().requires_grad_(True)
        lp, ent, pn = _head64(torch, z, v, a)
        (-ec * ent).sum().div(n).backward()
        with torch.no_grad():
            lr = lp - old[c0:c1].double()
            ratio = torch.exp(lr)
            A = adv[c0:c1].double()
            s1, s2 = ratio * A, ratio.clamp(1 - clip, 1 + clip) * A
            surr = torch.min(s1, s2)
            d = values[c0:c1].double() - ret[c0:c1].double()
            terms[:, c0:c1] = torch.stack([-surr, d * d, ent, (ratio - 1) - lr, ((ratio - 1).abs() > clip).double()])
            pa = pn.gather(1, a[:, None])[:, 0]
            # the gradient flows through min(s1, s2) where s1 is the minimum or the clip is inactive
            inside = (ratio >= 1 - clip) & (ratio <= 1 + clip)
            on = ((s1 < s2) | inside) & (pa >= EPS) & (pa <= 1 - EPS)
            amb_ratio = ((ratio - (1 - clip)).abs() < 2 ** -14) | ((ratio - (1 + clip)).abs() < 2 ** -14)
            n_amb += int(amb_ratio.sum())
            g_lp = (-A * ratio / n)[:, None] * _logp_grad64(torch, pn, a)
            r = _ref(torch, logits[c0:c1].double(), v)
            rtol, atol = _grad_tol(torch, dtype, A.abs() * ratio / n, torch.full_like(A, ec / n), r["H"], r["logS"])
            flipped += _check_grad(torch, dl[c0:c1], z.grad, g_lp, on, amb_ratio | _near_clamp(pa), rtol, atol, "dlogits")
            assert (dl[c0:c1][~v] == 0).all(), "nonzero gradient on a masked action"
            want_dv = 2 * vc * d / n
            assert ((dv[c0:c1].double() - want_dv).abs() <= 2.0 ** -22 * want_dv.abs()).all(), "dvalue"
    print("n=%d %s: %d rows at the clip or clamp edge took the other side" % (n, dtype, flipped))
    got = sums.cpu().numpy()
    want = terms.sum(1).cpu().numpy()
    scale = terms.abs().sum(1).cpu().numpy()
    for k in range(4):
        assert abs(got[k] - want[k]) <= 2.0 ** -15 * scale[k], (k, got[k], want[k], scale[k])
    assert abs(got[4] - want[4]) <= n_amb, (got[4], want[4], n_amb)
    assert 0.05 * n < want[4] < 0.95 * n                    # both branches of the clipped minimum are exercised
