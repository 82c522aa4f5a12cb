"""K5, the fused BatchNorm + ReLU (+ residual add) kernels of csrc/bb_bn_kernels.cu, against float64 references on
[M, C] bf16 activations: at the PPO minibatch and rollout sizes, and at every trip boundary of the kernels'
grid-stride loops.

Launch geometry (bb_launch_bn_relu_fwd / _bwd).  A thread owns one 8-channel group of G = C/8 and one of R = 256/G
row lanes of its block; need = ceil(M/R) blocks would give every thread one row.  The reduce grid is
min(need, 8 SMs), the apply grid min(max(ceil(need/4), 1), 8 SMs) with U = 4 rows in flight, the dx grid the same
with U = 3 (no skip) or U = 2 (skip).  With a capped grid one trip covers S = 8 SMs R rows, and a thread of the
reduce accumulates k = ceil(M / (reduce grid R)) rows.  S, R and k are computed from the device's SM count.

u = 2^-24 (half an fp32 ulp, relative).  A sum of n terms added one by one in fp32 is within (n - 1) u sum|terms|
of the exact sum.  A reduction adds k rows per thread, then R row lanes per block in fp32; the finalize adds the
block partials in double (2^-53, negligible).  So every per-channel sum is within (k + R) u sum|terms|.

Forward statistics.  The reduce sums d = x - K and d^2, K = x[row 0] of the channel; mean = K + s/M,
var = q/M - (s/M)^2 in double.  x - K adds at most u |d|.
- mean: |mean - mean64| <= (k + R + 1) u mean|x - K| + u |mean| (the fp32 store)
  <= (k + R + 2) u max(mean|x|, mean|x - K|), which also bounds an unshifted sum.
- rstd: |rstd / rstd64 - 1| <= 2^-14 on every channel.  This is a requirement, not a rounding bound: it is 32x
  below the 2^-9 resolution of the bf16 output, so the statistics cannot move y by more than 1/32 of its ulp,
  and it is above the 1.4e-5 an unshifted single-pass sum reaches at mean = 100 sigma.  A constant channel has
  var64 = 0 and must give float32(1/sqrt(eps)) within 2 ulp.
- on integers in [-8, 8] every fp32 partial of both sums is an integer below 2^24, hence exact: save_mean equals
  float32(sum x / M) bit for bit and save_rstd is within 1 ulp of float32(1/sqrt(var64 + eps)).
- running statistics against the float64 momentum update (momentum m, pre_bias b, unbiased variance):
  |rm - rm64| <= m band_mean + 4u ((1 - m)|rm0| + m (|mean| + |b|)) for the five fp32 operations;
  |rv - rv64| <= m M/(M - 1) 2^-13 (var + eps) + 4u ((1 - m)|rv0| + m var_unbiased), where 2^-13 (var + eps) is
  the variance error that the rstd requirement allows.

Forward output.  sc = fp32(gamma rstd) and sf = fma_fp32(-mean, sc, beta) are formed exactly from the kernel's own
save_mean / save_rstd (rational arithmetic on the host).  The kernel's fma and the skip add round twice:
t = 3u (|x sc| + |sf| + |skip|) covers both; the bf16 store adds half an ulp, so
|y - relu(x sc + sf + skip)| <= hulp(|ref| + t) + t, hulp(v) = half a bf16 ulp in v's binade.
Eval mode: sc = gamma rsqrtf(rv + eps) carries rsqrtf's 2 ulp (4u) plus the add and the multiply (1.5u), and
sf = beta + (b - rm) sc three more roundings, so t = 12u (|x sc| + |(b - rm) sc| + |beta| + |skip|) against
sc64 = gamma / sqrt(rv + eps).

Backward.  The float64 reference uses the kernel's saved statistics, xhat = (x - mean) rstd, and the kernel's ReLU
mask: y > 0 with a skip input; without one the sign of x sc + sf in float64 (x sc is exact in float64 and a
rounding never changes a sign, so this is the sign of the kernel's fma).  g = dy mask.
- dbeta = sum g: (k + R + 2) u sum|g|; bit for bit float32(sum g) on integer dy in [-4, 4].
- dgamma = sum g xhat: the kernel's xhat has two roundings and the fma one more:
  (k + R + 4) u sum|g xhat|.
- dx = sc (g - c1 - xhat c2), c1 = dbeta/M, c2 = dgamma/M: the coefficients carry the two sums' bands plus a
  store, the expression five roundings: t = |sc| (dc1 + |xhat| dc2 + 5u (|g| + |c1| + |xhat c2|)), and
  |dx - dx64| <= hulp(|dx64| + t) + t.
- dskip = g bit for bit.

Every output is pre-filled with NaN and has 64 guard rows past M that must stay NaN, so a row the kernel never
writes, or writes past the end, fails.  The float64 references run on the device in chunks of 2^25 elements.
"""
import math
from fractions import Fraction

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
EPS = float(np.float32(1e-5))            # the kernel takes eps and momentum as float
MOM = float(np.float32(0.1))
THREADS = 256
GUARD = 64
CHUNK = 1 << 25
WORST = {}

BOUNDARY_C = [8, 24, 64, 128, 2040, 2048]
BOUNDARY_M = ["1", "7", "S-1", "S", "S+1", "3S+1", "4S-1", "4S+1", "4S+2999"]
MINIBATCH, TRAIN_DEMO, REF_SCHEDULE, ROLLOUT = 2097152, 524288, 131072, 262144    # 32,768 / 8,192 / 2,048 / 4,096 x 64


@pytest.fixture(scope="module")
def torch():
    import torch
    yield torch
    print("\nworst error as a fraction of its band:")
    for k in sorted(WORST):
        print("  %-28s %.3g" % (k, WORST[k]))


def _geom(torch, M, C):
    """(R, S, k): row lanes per block, rows per trip of the capped grid, rows one reduce thread accumulates."""
    R = THREADS // (C // 8)
    cap = 8 * torch.cuda.get_device_properties(0).multi_processor_count
    red = min(-(-M // R), cap)
    return R, cap * R, -(-M // (red * R))


def _rows(spec, S):
    if spec.startswith("4S"):
        return 4 * S + int(spec[2:])
    if spec.startswith("3S"):
        return 3 * S + int(spec[2:])
    if spec.startswith("S"):
        return S + int(spec[1:] or 0)
    return int(spec)


def _chunks(M, C):
    step = max(1, CHUNK // C)
    for c0 in range(0, M, step):
        yield c0, min(M, c0 + step)


def _nan(torch, shape, dtype=None):
    import torch as T
    return T.full(shape, float("nan"), dtype=dtype or T.float32, device="cuda")


def _hulp(torch, v):
    """half a bf16 ulp in the binade of |v| (0 at 0)."""
    _, e = torch.frexp(v)
    return torch.where(v == 0, torch.zeros_like(v), torch.ldexp(torch.ones_like(v), (e - 9).double()))


def _within(torch, what, err, band):
    ratio = torch.where(band > 0, err / band, torch.where(err > 0, torch.full_like(err, math.inf), torch.zeros_like(err)))
    ratio = torch.where(torch.isnan(err), torch.full_like(err, math.inf), ratio)
    worst = float(ratio.max()) if ratio.numel() else 0.0
    WORST[what] = max(WORST.get(what, 0.0), worst)
    if not worst <= 1.0:
        bad = torch.nonzero(~(ratio <= 1.0))[:5].tolist()
        raise AssertionError("%s outside its band: worst %.3g of the band at %s" % (what, worst, bad))


# ------------------------------------------------------------------------------------------------ data
def _int_data(torch, M, C, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randint(-8, 9, (M, C), device="cuda", generator=g).to(torch.bfloat16)
    dy = torch.randint(-4, 5, (M, C), device="cuda", generator=g).to(torch.bfloat16)
    skip = torch.randint(-4, 5, (M, C), device="cuda", generator=g).to(torch.bfloat16)
    return x, dy, skip


def _real_data(torch, M, C, seed):
    """Channel c has kind c % 8: N(0.4, 1.7); relu(N) + 0.75; sigma from 1e-3 to 1e2 at mean 0.4 sigma; the same
    sigmas at mean 100 sigma; constant 0 or 1.0078125; constant 11.6875; 11.6875 with six rows one bf16 ulp above
    (11.75, none of them row 0); N(-5, 1.7)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    n = max(C // 8, 1)
    x = torch.empty(M, C, dtype=torch.bfloat16, device="cuda")
    for c in range(C):
        kind, j = c % 8, c // 8
        sig = 10.0 ** (-3 + 5 * j / max(n - 1, 1))
        if kind in (4, 5, 6):
            x[:, c] = (0.0 if j % 2 == 0 else 1.0078125) if kind == 4 else 11.6875
            if kind == 6:
                x[[1, M // 3, M // 2, M // 2 + 1, M - 2, M - 1], c] = 11.75
            continue
        z = torch.randn(M, device="cuda", generator=g)
        x[:, c] = (0.4 + 1.7 * z, torch.relu(z) + 0.75, sig * (z + 0.4), sig * (z + 100.0), None, None, None,
                   1.7 * z - 5.0)[kind]
    dy = torch.randn(M, C, device="cuda", generator=g).to(torch.bfloat16)
    skip = torch.randn(M, C, device="cuda", generator=g).to(torch.bfloat16)
    return x, dy, skip


def _params(torch, C, seed):
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    gamma = torch.rand(C, device="cuda", generator=g) + 0.5
    beta = torch.randn(C, device="cuda", generator=g) * 0.3
    pb = torch.randn(C, device="cuda", generator=g)
    rm = torch.randn(C, device="cuda", generator=g) * 0.2
    rv = torch.rand(C, device="cuda", generator=g) + 0.5
    return gamma, beta, pb, rm, rv


# ------------------------------------------------------------------------------------------------ kernels
def _ws(torch, C):
    from bbgpu import capi
    return _nan(torch, (capi.bn_workspace_size(C),))


def _fwd(torch, x, skip, gamma, beta, pb, rm, rv, training=True):
    from bbgpu import capi
    M, C = x.shape
    y = _nan(torch, (M + GUARD, C), torch.bfloat16)
    sm, sr = _nan(torch, (C,)), _nan(torch, (C,))
    capi.bn_relu_forward(x, skip, gamma, beta, pb, rm, rv, 0.1, 1e-5, training, y[:M], sm, sr, _ws(torch, C), M, C)
    torch.cuda.synchronize()
    assert torch.isnan(y[M:].float()).all(), "forward wrote past row M"
    return y[:M], sm, sr


def _bwd(torch, x, y, dy, gamma, beta, sm, sr, with_y):
    """bn_relu_backward (mask from y, dskip written) or bn_relu_backward_no_skip (mask from x)."""
    from bbgpu import capi
    M, C = x.shape
    dx = _nan(torch, (M + GUARD, C), torch.bfloat16)
    dsk = _nan(torch, (M + GUARD, C), torch.bfloat16) if with_y else None
    dg, db = _nan(torch, (C,)), _nan(torch, (C,))
    if with_y:
        capi.bn_relu_backward(x, y, dy, gamma, sm, sr, dx[:M], dsk[:M], dg, db, _ws(torch, C), M, C)
    else:
        capi.bn_relu_backward_no_skip(x, dy, gamma, beta, sm, sr, dx[:M], dg, db, _ws(torch, C), M, C)
    torch.cuda.synchronize()
    assert torch.isnan(dx[M:].float()).all() and (dsk is None or torch.isnan(dsk[M:].float()).all()), \
        "backward wrote past row M"
    return dict(dx=dx[:M], dskip=None if dsk is None else dsk[:M], dgamma=dg, dbeta=db)


# ------------------------------------------------------------------------------------------------ references
def _f32(q):
    """The Fraction q rounded to the nearest float32, ties to even."""
    f = np.float32(float(q))
    cands = (np.nextafter(f, np.float32(-np.inf)), f, np.nextafter(f, np.float32(np.inf)))
    return min(cands, key=lambda c: (abs(Fraction(float(c)) - q), int(np.float32(c).view(np.uint32)) & 1))


def _affine(torch, gamma, beta, mean, rstd):
    """The kernel's sc = __fmul_rn(gamma, rstd) and sf = __fmaf_rn(-mean, sc, beta), exactly, as float64."""
    g, b, m, r = (t.double().cpu().numpy() for t in (gamma, beta, mean, rstd))
    sc = [_f32(Fraction(gi) * Fraction(ri)) for gi, ri in zip(g, r)]
    sf = [_f32(Fraction(bi) - Fraction(mi) * Fraction(float(si))) for bi, mi, si in zip(b, m, sc)]
    return (torch.tensor(np.array(sc, np.float64), device="cuda"), torch.tensor(np.array(sf, np.float64), device="cuda"))


def _stats64(torch, x):
    M, C = x.shape
    K = x[0].double()
    s = torch.zeros(C, dtype=torch.float64, device="cuda")
    sa, sk = s.clone(), s.clone()
    for c0, c1 in _chunks(M, C):
        xc = x[c0:c1].double()
        s += xc.sum(0)
        sa += xc.abs().sum(0)
        sk += (xc - K).abs().sum(0)
    mean = s / M
    v = torch.zeros_like(s)
    for c0, c1 in _chunks(M, C):
        v += (x[c0:c1].double() - mean).pow(2).sum(0)
    return dict(sum=s, mean=mean, var=v / M, abs=sa / M, absK=sk / M)


def _check_forward(torch, x, skip, gamma, beta, pb, rm0, rv0, rm, rv, y, sm, sr, exact):
    """Statistics, running statistics and y of a training-mode forward; returns the kernel's (sc, sf)."""
    M, C = x.shape
    R, S, k = _geom(torch, M, C)
    st = _stats64(torch, x)
    mean, var = st["mean"], st["var"]
    assert not torch.isnan(sm).any() and not torch.isnan(sr).any(), "save_mean / save_rstd not written"
    rstd32 = (1.0 / torch.sqrt(var + EPS)).float()
    ulp = (torch.nextafter(rstd32, torch.full_like(rstd32, math.inf)) - rstd32).double()
    err_r = (sr.double() - rstd32.double()).abs()
    if exact:
        assert torch.equal(sm, mean.float()), ("save_mean is not float32(sum x / M)", torch.nonzero(sm != mean.float())[:5])
        _within(torch, "int: save_rstd (ulp)", err_r, ulp)
        band_m = U * mean.abs()
    else:
        band_m = (k + R + 2) * U * torch.maximum(st["abs"], st["absK"])
        _within(torch, "mean", (sm.double() - mean).abs(), band_m)
        const = var == 0
        rstd64 = 1.0 / torch.sqrt(var + EPS)
        _within(torch, "rstd (2^-14)", ((sr.double() - rstd64).abs() / rstd64)[~const],
                torch.full_like(rstd64[~const], 2.0 ** -14))
        _within(torch, "rstd, constant channel (ulp)", err_r[const], 2 * ulp[const])
    # running statistics
    b = pb.double() if pb is not None else torch.zeros_like(mean)
    rm_ref = (1 - MOM) * rm0.double() + MOM * (mean + b)
    t_rm = MOM * band_m + 4 * U * ((1 - MOM) * rm0.double().abs() + MOM * (mean.abs() + b.abs()))
    _within(torch, "running_mean", (rm.double() - rm_ref).abs(), t_rm)
    unb = var * M / (M - 1) if M > 1 else var
    rv_ref = (1 - MOM) * rv0.double() + MOM * unb
    t_rv = MOM * (unb / var.clamp(min=1e-300)).clamp(min=1) * 2.0 ** -13 * (var + EPS) \
        + 4 * U * ((1 - MOM) * rv0.double().abs() + MOM * unb)
    _within(torch, "running_var", (rv.double() - rv_ref).abs(), t_rv)
    # y from the kernel's own affine pair
    sc, sf = _affine(torch, gamma, beta, sm, sr)
    for c0, c1 in _chunks(M, C):
        xs = x[c0:c1].double() * sc
        pre = xs + sf
        if skip is not None:
            pre = pre + skip[c0:c1].double()
        ref = torch.relu(pre)
        t = 3 * U * (xs.abs() + sf.abs() + (skip[c0:c1].double().abs() if skip is not None else 0))
        _within(torch, "y", (y[c0:c1].double() - ref).abs(), _hulp(torch, ref + t) + t)
    return sc, sf


def _check_backward(torch, x, dy, mask, gamma, sm, sr, sc, out, exact):
    """dgamma, dbeta, dx (and dskip) against float64 from the kernel's saved statistics; mask(c0, c1, x64)."""
    M, C = x.shape
    R, S, k = _geom(torch, M, C)
    mean, rstd = sm.double(), sr.double()
    z = torch.zeros(C, dtype=torch.float64, device="cuda")
    sg, sgx, sag, sagx = z.clone(), z.clone(), z.clone(), z.clone()
    for c0, c1 in _chunks(M, C):
        xc = x[c0:c1].double()
        xh = (xc - mean) * rstd
        g = torch.where(mask(c0, c1, xc), dy[c0:c1].double(), torch.zeros_like(xc))
        sg += g.sum(0)
        sgx += (g * xh).sum(0)
        sag += g.abs().sum(0)
        sagx += (g * xh).abs().sum(0)
        if out["dskip"] is not None:
            assert torch.equal(out["dskip"][c0:c1], g.to(torch.bfloat16)), ("dskip != dy * mask", c0)
    if exact:
        assert torch.equal(out["dbeta"], sg.float()), ("dbeta is not float32(sum dy * mask)",
                                                       torch.nonzero(out["dbeta"] != sg.float())[:5])
    else:
        _within(torch, "dbeta", (out["dbeta"].double() - sg).abs(), (k + R + 2) * U * sag)
    _within(torch, "dgamma", (out["dgamma"].double() - sgx).abs(), (k + R + 4) * U * sagx)
    c1_, c2_ = sg / M, sgx / M
    dc1, dc2 = (k + R + 2) * U * sag / M, (k + R + 4) * U * sagx / M
    for c0, c1 in _chunks(M, C):
        xc = x[c0:c1].double()
        xh = (xc - mean) * rstd
        g = torch.where(mask(c0, c1, xc), dy[c0:c1].double(), torch.zeros_like(xc))
        ref = sc * (g - c1_ - xh * c2_)
        t = sc.abs() * (dc1 + xh.abs() * dc2 + 5 * U * (g.abs() + c1_.abs() + (xh * c2_).abs()))
        _within(torch, "dx", (out["dx"][c0:c1].double() - ref).abs(), _hulp(torch, ref.abs() + t) + t)


def _case(torch, M, C, kind, seed, skip, pre_bias, backward=True):
    x, dy, s = (_int_data if kind == "int" else _real_data)(torch, M, C, seed)
    if not skip:
        s = None
    gamma, beta, pb, rm, rv = _params(torch, C, seed)
    if not pre_bias:
        pb = None
    rm0, rv0 = rm.clone(), rv.clone()
    y, sm, sr = _fwd(torch, x, s, gamma, beta, pb, rm, rv)
    sc, sf = _check_forward(torch, x, s, gamma, beta, pb, rm0, rv0, rm, rv, y, sm, sr, kind == "int")
    if not backward:
        return
    if skip:
        mask = lambda c0, c1, xc: y[c0:c1] > 0                  # noqa: E731
    else:
        mask = lambda c0, c1, xc: xc * sc + sf > 0              # noqa: E731
    out = _bwd(torch, x, y, dy, gamma, beta, sm, sr, with_y=skip)
    _check_backward(torch, x, dy, mask, gamma, sm, sr, sc, out, kind == "int")


# ------------------------------------------------------------------------------------------------ tests
@pytest.mark.parametrize("spec", BOUNDARY_M)
@pytest.mark.parametrize("C", BOUNDARY_C)
def test_trip_boundaries_are_exact_on_integer_data(torch, C, spec):
    """At G = 1 (C = 8), R = 85 with an idle thread (C = 24), R = 1 with an idle thread (C = 2040) and R = 1 with
    G = 256 (C = 2048), on rows around one trip S and four trips 4S (one thread's second row, a partial U-trip):
    forward statistics bit for bit, running statistics, y, and both backward variants with dbeta and dskip bit
    for bit."""
    R, S, _ = _geom(torch, 1, C)
    M = _rows(spec, S)
    _case(torch, M, C, "int", seed=C * 31 + len(spec), skip=True, pre_bias=True)
    _case(torch, M, C, "int", seed=C * 37 + len(spec), skip=False, pre_bias=False)


PRODUCTION = [(MINIBATCH, 64), (MINIBATCH, 128), (TRAIN_DEMO, 128), (REF_SCHEDULE, 128), (ROLLOUT, 64)]


@pytest.mark.parametrize("M,C", PRODUCTION)
def test_production_shapes_are_exact_on_integer_data(torch, M, C):
    _case(torch, M, C, "int", seed=M % 997 + C, skip=True, pre_bias=True)
    _case(torch, M, C, "int", seed=M % 991 + C, skip=False, pre_bias=False)


@pytest.mark.parametrize("skip", [True, False])
@pytest.mark.parametrize("M,C", [(MINIBATCH, 64), (MINIBATCH, 128), (TRAIN_DEMO, 128), (REF_SCHEDULE, 128)])
def test_training_step_matches_float64(torch, M, C, skip):
    """Forward (with pre_bias) and backward at the minibatch sizes of a 32,768-, 8,192- and 2,048-sample update,
    on real-valued channels including constant and near-constant ones."""
    _case(torch, M, C, "real", seed=M % 1009 + C + skip, skip=skip, pre_bias=True)


def test_rollout_forward_matches_float64(torch):
    """The first layer of a 4,096-env rollout forward: 262,144 x 64, training mode, no skip."""
    _case(torch, ROLLOUT, 64, "real", seed=77, skip=False, pre_bias=True, backward=False)


def test_eval_mode_matches_float64(torch):
    """Eval mode uses the running statistics (and pre_bias) and leaves them alone."""
    M, C = ROLLOUT, 128
    x, _, s = _real_data(torch, M, C, 5)
    gamma, beta, pb, rm, rv = _params(torch, C, 5)
    rm0, rv0 = rm.clone(), rv.clone()
    y, _, _ = _fwd(torch, x, s, gamma, beta, pb, rm, rv, training=False)
    assert torch.equal(rm, rm0) and torch.equal(rv, rv0), "eval mode changed the running statistics"
    sc = gamma.double() / torch.sqrt(rv.double() + EPS)
    bs = (pb.double() - rm.double()) * sc
    sf = beta.double() + bs
    for c0, c1 in _chunks(M, C):
        xs = x[c0:c1].double() * sc
        sk = s[c0:c1].double()
        ref = torch.relu(xs + sf + sk)
        t = 12 * U * (xs.abs() + bs.abs() + beta.double().abs() + sk.abs())
        _within(torch, "eval y", (y[c0:c1].double() - ref).abs(), _hulp(torch, ref + t) + t)


@pytest.mark.parametrize("C", [64, 128])
def test_backward_with_and_without_y_are_bit_identical(torch, C):
    """Without a residual input the backward recomputes the ReLU mask from x; at 2,097,152 rows it must give the
    gradients that reading the mask from the forward's y gives, bit for bit."""
    M = MINIBATCH
    x, dy, _ = _real_data(torch, M, C, 11)
    gamma, beta, pb, rm, rv = _params(torch, C, 11)
    y, sm, sr = _fwd(torch, x, None, gamma, beta, pb, rm, rv)
    a = _bwd(torch, x, y, dy, gamma, beta, sm, sr, with_y=True)
    b = _bwd(torch, x, y, dy, gamma, beta, sm, sr, with_y=False)
    for key in ("dx", "dgamma", "dbeta"):
        assert torch.equal(a[key], b[key]), key
    assert torch.equal(a["dskip"], torch.where(y > 0, dy, torch.zeros_like(dy)))


def test_two_calls_are_bit_identical(torch):
    """Fixed-order reductions: two identical forward and backward calls at 2,097,152 x 128 give the same bits,
    running statistics included."""
    M, C = MINIBATCH, 128
    x, dy, s = _real_data(torch, M, C, 13)
    gamma, beta, pb, rm, rv = _params(torch, C, 13)
    runs = []
    for _ in range(2):
        rm1, rv1 = rm.clone(), rv.clone()
        y, sm, sr = _fwd(torch, x, s, gamma, beta, pb, rm1, rv1)
        o1 = _bwd(torch, x, y, dy, gamma, beta, sm, sr, with_y=True)
        o2 = _bwd(torch, x, y, dy, gamma, beta, sm, sr, with_y=False)
        runs.append([y, sm, sr, rm1, rv1] + [o[k] for o in (o1, o2) for k in ("dx", "dgamma", "dbeta")] + [o1["dskip"]])
    for i, (p, q) in enumerate(zip(*runs)):
        assert torch.equal(p, q), i


def test_fused_bn_relu_wrapper_matches_float64(torch):
    """network.FusedBNReLU at (32,768, 128, 8, 8) with skip and pre_bias: channels-last activations, an
    NCHW-contiguous upstream gradient (the wrapper converts it), checked against the same float64 references."""
    from bbgpu.network import FusedBNReLU
    N, C, H, W = 32768, 128, 8, 8
    M = N * H * W
    x2, dy2, s2 = _real_data(torch, M, C, 17)
    gamma, beta, pb, rm, rv = _params(torch, C, 17)
    rm0, rv0 = rm.clone(), rv.clone()

    def nchw(t):
        return t.view(N, H, W, C).permute(0, 3, 1, 2)

    x = nchw(x2).detach().requires_grad_(True)
    s = nchw(s2).detach().requires_grad_(True)
    g = gamma.clone().requires_grad_(True)
    b = beta.clone().requires_grad_(True)
    assert x.is_contiguous(memory_format=torch.channels_last)
    y = FusedBNReLU.apply(x, s, g, b, rm, rv, True, 0.1, 1e-5, pb)
    sm, sr = y.grad_fn.saved_tensors[3], y.grad_fn.saved_tensors[4]
    y2 = y.detach().permute(0, 2, 3, 1).reshape(M, C)
    sc, _ = _check_forward(torch, x2, s2, gamma, beta, pb, rm0, rv0, rm, rv, y2, sm, sr, False)
    gy = nchw(dy2).contiguous()
    del dy2
    assert gy.is_contiguous() and not gy.is_contiguous(memory_format=torch.channels_last)
    y.backward(gy)
    dy_rows = gy.permute(0, 2, 3, 1).contiguous().view(M, C)
    del gy
    out = dict(dx=x.grad.permute(0, 2, 3, 1).reshape(M, C), dskip=s.grad.permute(0, 2, 3, 1).reshape(M, C),
               dgamma=g.grad, dbeta=b.grad)
    _check_backward(torch, x2, dy_rows, lambda c0, c1, xc: y2[c0:c1] > 0, gamma, sm, sr, sc, out, False)
