"""GPU parity tests for K2 (obs unpack), K3 (masked sample) and K4 (GAE)."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


# ------------------------------------------------------------------ K4
@pytest.mark.parametrize("T,N", [(128, 4096), (16, 8), (1, 3), (33, 1001), (128, 64), (7, 4)])
def test_gae_bit_exact_with_oracle(torch, T, N):
    from bbgpu import capi
    from oracle import bb_oracle_c as OC
    rs = np.random.RandomState(T * 1000 + N)
    r = (rs.randn(T, N) * 2).astype(np.float32)
    v = rs.randn(T, N).astype(np.float32)
    d = (rs.rand(T, N) < 0.1).astype(np.float32)
    lv = rs.randn(N).astype(np.float32)
    want_a, want_r = OC.gae(r, v, d, lv, 0.99, 0.95)
    tr, tv, td, tl = (torch.from_numpy(x).cuda() for x in (r, v, d, lv))
    adv, ret = torch.empty_like(tr), torch.empty_like(tr)
    mom = torch.zeros(2, dtype=torch.float64, device="cuda")
    capi.gae(tr, tv, td, tl, 0.99, 0.95, adv, ret, mom)
    torch.cuda.synchronize()
    assert np.array_equal(adv.cpu().numpy().view(np.uint32), want_a.view(np.uint32))
    assert np.array_equal(ret.cpu().numpy().view(np.uint32), want_r.view(np.uint32))
    m = mom.cpu().numpy()
    np.testing.assert_allclose(m[0], want_a.astype(np.float64).sum(), rtol=1e-9, atol=1e-6)
    np.testing.assert_allclose(m[1], (want_a.astype(np.float64) ** 2).sum(), rtol=1e-9)


def test_gae_matches_reference_golden(torch):
    from bbgpu import capi
    g = np.load(os.path.join(G, "gae_golden.npz"))
    for tag in "abc":
        tr, tv, td, tl = (torch.from_numpy(g[f"{tag}_{k}"]).cuda() for k in ("rewards", "values", "dones", "last"))
        adv, ret = torch.empty_like(tr), torch.empty_like(tr)
        capi.gae(tr, tv, td, tl, float(g["gamma"]), float(g["lam"]), adv, ret, None)
        torch.cuda.synchronize()
        # north_star tolerance is 1e-5 relative; the kernel is in fact bit-identical
        np.testing.assert_allclose(adv.cpu().numpy(), g[f"{tag}_adv"], rtol=1e-5, atol=0)
        assert np.array_equal(adv.cpu().numpy(), g[f"{tag}_adv"]) and np.array_equal(ret.cpu().numpy(), g[f"{tag}_ret"])


# ------------------------------------------------------------------ K2
def test_unpack_obs_matches_reference_layout(torch):
    from bbgpu import capi, vec_env
    n = 3000
    h = capi.EnvHandle(n, 8)
    h.step_random(25)
    board = torch.zeros(n, dtype=torch.int64, device="cuda")
    pieces = torch.zeros(n, dtype=torch.int32, device="cuda")
    mask = torch.zeros((3, n), dtype=torch.int64, device="cuda")
    h.observe(board, pieces, mask)
    obs32 = torch.empty((n, 4, 8, 8), dtype=torch.float32, device="cuda")
    obs16 = torch.empty((n, 4, 8, 8), dtype=torch.bfloat16, device="cuda")
    m8 = torch.empty((n, 192), dtype=torch.uint8, device="cuda")
    m32 = torch.empty((n, 192), dtype=torch.float32, device="cuda")
    capi.unpack_obs(board, pieces, mask, n, obs=obs32, mask_dense=m8)
    capi.unpack_obs(board, pieces, mask, n, obs=obs16, mask_dense=m32)
    torch.cuda.synchronize()
    b = board.cpu().numpy().view(np.uint64)
    p = pieces.cpu().numpy().view(np.uint32)
    m = mask.cpu().numpy().view(np.uint64)
    want_board = vec_env.expand_board(b)
    want_pieces = vec_env.expand_pieces(p)
    want_mask = vec_env.expand_mask(m)
    o = obs32.cpu().numpy()
    assert np.array_equal(o[:, 0], want_board) and np.array_equal(o[:, 1:], want_pieces)
    assert np.array_equal(obs16.float().cpu().numpy(), o)
    assert np.array_equal(m8.cpu().numpy(), want_mask.astype(np.uint8))
    assert np.array_equal(m32.cpu().numpy(), want_mask.astype(np.float32))
    # cross-check the numpy expansion itself against the cell oracle on a few envs
    from oracle import bb_oracle as O
    for i in range(0, n, 211):
        g = np.array(O.u64_to_grid(int(b[i])), dtype=np.float32)
        assert np.array_equal(want_board[i], g)
        for k in range(3):
            pid, used = (int(p[i]) >> (8 * k)) & 0xFF, (int(p[i]) >> (24 + k)) & 1
            plane = np.zeros((8, 8), np.float32)
            if not used:
                for dr, dc in O.PIECE_CELLS[pid]:
                    plane[dr, dc] = 1
            assert np.array_equal(want_pieces[i, k], plane)
    h.close()


# ------------------------------------------------------------------ K3
def _planes_from_dense(mask_dense):
    n = mask_dense.shape[0]
    packed = np.packbits(mask_dense.astype(np.uint8).reshape(n, 24, 8), axis=2, bitorder="little").reshape(n, 24)
    return np.ascontiguousarray(packed.view(np.uint64).reshape(n, 3).T)


def test_masked_head_matches_reference_golden(torch):
    from bbgpu import capi
    g = np.load(os.path.join(G, "policy_golden.npz"))
    n = g["logits"].shape[0]
    logits = torch.from_numpy(g["logits"]).cuda().contiguous()
    planes = torch.from_numpy(_planes_from_dense(g["mask"]).view(np.int64)).cuda()
    act = torch.from_numpy(g["actions"].astype(np.int32)).cuda()
    logp = torch.empty(n, dtype=torch.float32, device="cuda")
    ent = torch.empty(n, dtype=torch.float32, device="cuda")
    capi.masked_sample(logits, planes, n, 0, 0, 2, act, logp, ent)          # evaluate given actions
    torch.cuda.synchronize()
    np.testing.assert_allclose(logp.cpu().numpy(), g["log_prob"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(ent.cpu().numpy(), g["entropy"], rtol=1e-5, atol=1e-6)
    act2 = torch.zeros(n, dtype=torch.int32, device="cuda")
    capi.masked_sample(logits, planes, n, 0, 0, 1, act2, logp, ent)         # deterministic
    torch.cuda.synchronize()
    assert np.array_equal(act2.cpu().numpy(), g["argmax"])
    np.testing.assert_allclose(logp.cpu().numpy(), g["log_prob_argmax"], rtol=1e-5, atol=1e-6)


def test_masked_head_vs_oracle_random_rows(torch):
    from bbgpu import capi
    from oracle import bb_oracle as O
    rs = np.random.RandomState(4)
    n = 5000
    logits = (rs.randn(n, 192) * 4).astype(np.float32)
    dense = rs.rand(n, 192) < rs.rand(n, 1) * 0.5
    dense[np.arange(n), rs.randint(0, 192, n)] = True          # at least one valid action
    dense[0] = False; dense[0, 191] = True                      # single valid action
    dense[1] = True                                             # everything valid
    acts = (rs.rand(n, 192) * dense).argmax(1).astype(np.int32)
    acts[2] = int(np.where(~dense[2])[0][0]) if (~dense[2]).any() else acts[2]   # an INVALID action
    probs, want_lp, want_ent = O.masked_policy_terms(logits, dense, acts)
    tl = torch.from_numpy(logits).cuda()
    planes = torch.from_numpy(_planes_from_dense(dense).view(np.int64)).cuda()
    ta = torch.from_numpy(acts).cuda()
    lp = torch.empty(n, dtype=torch.float32, device="cuda")
    en = torch.empty(n, dtype=torch.float32, device="cuda")
    capi.masked_sample(tl, planes, n, 0, 0, 2, ta, lp, en)
    torch.cuda.synchronize()
    np.testing.assert_allclose(lp.cpu().numpy(), want_lp, rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(en.cpu().numpy(), want_ent, rtol=2e-5, atol=2e-6)
    # bf16 logits: same maths on the rounded inputs
    tb = tl.bfloat16()
    _, want_lp16, want_ent16 = O.masked_policy_terms(tb.float().cpu().numpy(), dense, acts)
    capi.masked_sample(tb.contiguous(), planes, n, 0, 0, 2, ta, lp, en)
    torch.cuda.synchronize()
    np.testing.assert_allclose(lp.cpu().numpy(), want_lp16, rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(en.cpu().numpy(), want_ent16, rtol=2e-5, atol=2e-6)


def test_sampling_is_valid_reproducible_and_distributed_like_softmax(torch):
    """Sampling cannot be bit-matched to torch.multinomial (SURVEY §7.3): check that every
    sample is a valid action, the Philox stream is reproducible and matches the host
    replica's inverse CDF, and frequencies pass a chi-square test."""
    from bbgpu import capi, philox
    from oracle import bb_oracle as O
    rs = np.random.RandomState(6)
    n = 200000
    row_logits = (rs.randn(192) * 1.5).astype(np.float32)
    row_mask = rs.rand(192) < 0.3
    row_mask[5] = True
    logits = torch.from_numpy(np.tile(row_logits, (n, 1))).cuda()
    dense = np.tile(row_mask, (n, 1))
    planes = torch.from_numpy(_planes_from_dense(dense).view(np.int64)).cuda()
    a1 = torch.zeros(n, dtype=torch.int32, device="cuda")
    a2 = torch.zeros(n, dtype=torch.int32, device="cuda")
    lp = torch.empty(n, dtype=torch.float32, device="cuda")
    capi.masked_sample(logits, planes, n, 99, 7, 0, a1, lp, None)
    capi.masked_sample(logits, planes, n, 99, 7, 0, a2, None, None)
    torch.cuda.synchronize()
    s = a1.cpu().numpy()
    assert np.array_equal(s, a2.cpu().numpy())
    assert row_mask[s].all()
    probs, _, _ = O.masked_policy_terms(row_logits[None], row_mask[None], np.array([5]))
    probs = probs[0].astype(np.float64)
    # host replica of the inverse CDF (same uniforms, the kernel's documented action order)
    u = philox.sample_uniforms(99, 7, n).astype(np.float64)
    order = philox.sample_order()
    assert sorted(order.tolist()) == list(range(192))
    cdf = np.cumsum(probs[order])
    host = order[np.minimum(np.searchsorted(cdf, u * cdf[-1], side="right"), 191)]
    assert (host == s).mean() > 0.9995        # float32 vs float64 prefix sums may differ at bin edges
    cnt = np.bincount(s, minlength=192)[row_mask].astype(np.float64)
    exp = probs[row_mask] / probs[row_mask].sum() * n
    keep = exp > 5
    chi2 = ((cnt[keep] - exp[keep]) ** 2 / exp[keep]).sum()
    dof = keep.sum() - 1
    assert chi2 < dof + 6 * np.sqrt(2 * dof), (chi2, dof)
    # log-prob of the sampled action is log p[a]
    np.testing.assert_allclose(lp.cpu().numpy(), np.log(probs[s]).astype(np.float32), rtol=1e-4, atol=1e-5)
    # a different call counter gives a different draw
    capi.masked_sample(logits, planes, n, 99, 8, 0, a2, None, None)
    torch.cuda.synchronize()
    assert (a2.cpu().numpy() != s).mean() > 0.5


@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
def test_masked_head_backward_kernel_matches_torch_autograd(torch, dtype):
    """K3 in evaluate mode (log-prob, entropy) and bb_masked_head_backward against autograd through
    the torch restatement of network.py:210-262 (which tests/test_ppo_host.py pins to the reference)."""
    from bbgpu import capi
    from bbgpu.network import _pack_mask_planes
    torch.manual_seed(3)
    n = 4096
    dt = getattr(torch, dtype)
    base = (torch.randn(n, 192, device="cuda") * 3).to(dt)
    dense = (torch.rand(n, 192, device="cuda") < torch.rand(n, 1, device="cuda") * 0.6)
    dense[torch.arange(n), torch.randint(0, 192, (n,))] = True
    dense[0] = False; dense[0, 17] = True                       # single valid action: p = 1 -> clamp kills the gradient
    act = (torch.rand(n, 192, device="cuda") * dense).argmax(1)
    w1, w2 = torch.randn(n, device="cuda"), torch.randn(n, device="cuda")
    planes = _pack_mask_planes(dense)

    def ref(logits):
        probs = torch.softmax(logits.float().masked_fill(~dense, float("-inf")), -1)
        eps = torch.finfo(torch.float32).eps
        pn = probs / probs.sum(-1, keepdim=True)
        lp = torch.log(pn.clamp(eps, 1 - eps)).gather(1, act.unsqueeze(1)).squeeze(1)
        q = probs / probs.sum(-1, keepdim=True).clamp(min=1e-10)
        ent = -(q * torch.log(q.clamp(min=1e-10)) * dense).sum(-1)
        return lp, ent

    a = base.clone().requires_grad_(True)
    lp_r, en_r = ref(a)
    (w1 * lp_r + w2 * en_r).sum().backward()
    act32 = act.to(torch.int32)
    lp_f, en_f = torch.empty(n, device="cuda"), torch.empty(n, device="cuda")
    capi.masked_sample(base, planes, planes.stride(0), 0, 0, 2, act32, lp_f, en_f)
    grad = torch.empty_like(base)                                # d(w1 . logp + w2 . entropy) / d logits
    capi.masked_head_backward(base, planes, planes.stride(0), act32, w1, w2, grad)
    torch.testing.assert_close(lp_f, lp_r, rtol=1e-5, atol=2e-6)
    torch.testing.assert_close(en_f, en_r, rtol=1e-5, atol=2e-6)
    tol = dict(rtol=2e-2, atol=2e-2) if dtype == "bfloat16" else dict(rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(grad.float(), a.grad.float(), **tol)
    assert (grad[~dense] == 0).all() and grad.dtype == dt
    assert float(grad[0].abs().sum()) == 0.0                     # clamped at 1 - eps, like torch


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
def test_fused_ppo_loss_tail_matches_torch(torch, dtype):
    """bb_ppo_loss (PPOLossTail) against the torch statement of src/agents/ppo.py:366-395 on top of
    network.py:210-262: loss, the five metric means, d loss/d logits and d loss/d values."""
    from bbgpu.network import PPOLossTail, _pack_mask_planes
    torch.manual_seed(11)
    n, clip, vc, ec = 6000, 0.2, 0.5, 0.01
    dt = getattr(torch, dtype)
    base = (torch.randn(n, 192, device="cuda") * 2).to(dt)
    dense = (torch.rand(n, 192, device="cuda") < torch.rand(n, 1, device="cuda") * 0.6)
    dense[torch.arange(n), torch.randint(0, 192, (n,))] = True
    dense[0] = False; dense[0, 5] = True
    act = (torch.rand(n, 192, device="cuda") * dense).argmax(1)
    planes = _pack_mask_planes(dense)
    values0 = torch.randn(n, device="cuda")
    ret = values0 + torch.randn(n, device="cuda")
    adv = torch.randn(n, device="cuda")
    eps = torch.finfo(torch.float32).eps

    def head(logits):
        probs = torch.softmax(logits.float().masked_fill(~dense, float("-inf")), -1)
        pn = probs / probs.sum(-1, keepdim=True)
        lp = torch.log(pn.clamp(eps, 1 - eps)).gather(1, act.unsqueeze(1)).squeeze(1)
        q = probs / probs.sum(-1, keepdim=True).clamp(min=1e-10)
        return lp, -(q * torch.log(q.clamp(min=1e-10)) * dense).sum(-1)

    with torch.no_grad():                                   # old policy = perturbed current one -> ratios on both sides of the clip
        old_logp = head(base)[0] + 0.25 * torch.randn(n, device="cuda")
    a, va = base.clone().requires_grad_(True), values0.clone().requires_grad_(True)
    lp, ent = head(a)
    ratio = torch.exp(lp - old_logp)
    pl = -torch.min(ratio * adv, torch.clamp(ratio, 1 - clip, 1 + clip) * adv).mean()
    vl = torch.nn.functional.mse_loss(va, ret)
    loss_r = pl + vc * vl - ec * ent.mean()
    loss_r.backward()
    kl = ((ratio - 1) - torch.log(ratio)).mean()
    cf = ((ratio - 1).abs() > clip).float().mean()

    b, vb = base.clone().requires_grad_(True), values0.clone().requires_grad_(True)
    loss_f, means = PPOLossTail.apply(b, vb, planes, act, old_logp, adv, ret, clip, vc, ec)
    (3.0 * loss_f).backward()                               # the incoming gradient is applied
    ref_means = torch.stack([pl, vl, ent.mean(), kl, cf]).double()
    torch.testing.assert_close(means, ref_means.detach(), rtol=2e-5, atol=2e-6)
    torch.testing.assert_close(loss_f, loss_r.detach(), rtol=2e-5, atol=2e-6)
    tol = dict(rtol=2e-2, atol=2e-5) if dtype == "bfloat16" else dict(rtol=2e-4, atol=2e-8)
    torch.testing.assert_close(b.grad.float() / 3.0, a.grad.float(), **tol)
    torch.testing.assert_close(vb.grad / 3.0, va.grad, rtol=1e-5, atol=1e-9)
    assert (b.grad[~dense] == 0).all() and b.grad.dtype == dt and not means.requires_grad
    frac_clipped = float(cf)
    assert 0.05 < frac_clipped < 0.95                      # the test exercises both branches of the min


@pytest.mark.gpu
@pytest.mark.parametrize("shape,with_skip", [((96, 64, 8, 8), False), ((64, 128, 8, 8), True), ((7, 128, 8, 8), True),
                                             ((33, 24, 3, 5), False),
                                             ((320, 64, 8, 8), True), ((288, 128, 8, 8), False)])
def test_fused_bn_relu_matches_torch(torch, shape, with_skip):
    """bb_bn_relu_forward/backward (FusedBNReLU) against torch's batch_norm (+ skip) + relu with
    autograd, both on bf16 channels-last activations (network.py:14-31, 78-92), incl. the running
    statistics update and eval mode."""
    import torch.nn.functional as F
    from bbgpu.network import FusedBNReLU
    torch.manual_seed(5)
    n, c, h, w = shape
    x0 = (torch.randn(shape, device="cuda") * 1.7 + 0.4).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    s0 = torch.randn(shape, device="cuda").to(torch.bfloat16).contiguous(memory_format=torch.channels_last) if with_skip else None
    gamma0, beta0 = torch.rand(c, device="cuda") + 0.5, torch.randn(c, device="cuda") * 0.3
    gy = torch.randn(shape, device="cuda").to(torch.bfloat16).contiguous(memory_format=torch.channels_last)

    def run(fused):
        x = x0.clone().requires_grad_(True)
        s = s0.clone().requires_grad_(True) if with_skip else None
        g, b = gamma0.clone().requires_grad_(True), beta0.clone().requires_grad_(True)
        rm, rv = torch.zeros(c, device="cuda"), torch.ones(c, device="cuda")
        if fused:
            y = FusedBNReLU.apply(x, s, g, b, rm, rv, True, 0.1, 1e-5)
        else:                                       # fp32 maths on the same bf16 inputs = the exact answer
            z = F.batch_norm(x.float(), rm, rv, g, b, True, 0.1, 1e-5)
            if with_skip:
                z = z + s.float()
            y = F.relu(z)
        y.backward(gy.to(y.dtype))
        return y.detach().float(), x.grad.float(), (s.grad.float() if with_skip else None), g.grad, b.grad, rm, rv

    yf, dxf, dsf, dgf, dbf, rmf, rvf = run(True)
    yr, dxr, dsr, dgr, dbr, rmr, rvr = run(False)
    torch.testing.assert_close(yf, yr, rtol=1e-2, atol=1e-2)                       # bf16 output rounding
    torch.testing.assert_close(rmf, rmr, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(rvf, rvr, rtol=1e-4, atol=1e-6)
    # the relu mask comes from the bf16 output: entries with |y| below bf16 resolution may flip, so
    # compare the gradients in aggregate and elementwise with a small budget of mismatches
    bad = ((dxf - dxr).abs() > 2e-2 + 2e-2 * dxr.abs()).float().mean()
    assert float(bad) < 2e-3
    torch.testing.assert_close(dgf, dgr, rtol=2e-2, atol=2e-2 * float(dgr.abs().max()))
    torch.testing.assert_close(dbf, dbr, rtol=2e-2, atol=2e-2 * float(dbr.abs().max()))
    if with_skip:
        assert float(((dsf - dsr).abs() > 1e-2).float().mean()) < 2e-3
    # eval mode uses the running statistics and leaves them alone
    rm, rv = torch.randn(c, device="cuda") * 0.2, torch.rand(c, device="cuda") + 0.5
    rm0, rv0 = rm.clone(), rv.clone()
    with torch.no_grad():
        ye = FusedBNReLU.apply(x0, s0, gamma0, beta0, rm, rv, False, 0.1, 1e-5).float()
        ze = F.batch_norm(x0.float(), rm, rv, gamma0, beta0, False, 0.1, 1e-5)
        ze = F.relu(ze + s0.float()) if with_skip else F.relu(ze)
    torch.testing.assert_close(ye, ze, rtol=1e-2, atol=1e-2)
    assert torch.equal(rm, rm0) and torch.equal(rv, rv0)
    # pre_bias = a conv bias left out of x: cancels in the training output, is tracked by the running
    # mean, and is applied in eval mode — i.e. identical to batch_norm(x + bias)
    pb = torch.randn(c, device="cuda")
    rm1, rv1 = torch.zeros(c, device="cuda"), torch.ones(c, device="cuda")
    rm2, rv2 = torch.zeros(c, device="cuda"), torch.ones(c, device="cuda")
    with torch.no_grad():
        y1 = FusedBNReLU.apply(x0, s0, gamma0, beta0, rm1, rv1, True, 0.1, 1e-5, pb).float()
        z2 = F.batch_norm(x0.float() + pb.view(1, -1, 1, 1), rm2, rv2, gamma0, beta0, True, 0.1, 1e-5)
        z2 = F.relu(z2 + s0.float()) if with_skip else F.relu(z2)
        torch.testing.assert_close(y1, z2, rtol=1e-2, atol=1e-2)
        torch.testing.assert_close(rm1, rm2, rtol=1e-5, atol=1e-5)
        torch.testing.assert_close(rv1, rv2, rtol=1e-4, atol=1e-6)
        y3 = FusedBNReLU.apply(x0, s0, gamma0, beta0, rm, rv, False, 0.1, 1e-5, pb).float()
        z3 = F.batch_norm(x0.float() + pb.view(1, -1, 1, 1), rm, rv, gamma0, beta0, False, 0.1, 1e-5)
        z3 = F.relu(z3 + s0.float()) if with_skip else F.relu(z3)
        torch.testing.assert_close(y3, z3, rtol=1e-2, atol=2e-2)


@pytest.mark.gpu
def test_network_with_fused_bn_matches_torch_path(torch):
    """The whole trunk with FusedBNReLU, bf16 autocast + channels-last as PPOAgent(precision='bf16')
    runs it.  Two bf16 pipelines differ from each other by their rounding noise, so both are
    measured against the fp32 network with the same weights: the fused path must be as close to it
    as torch's own bf16 path (outputs, parameter gradients, BatchNorm buffers)."""
    import copy
    from bbgpu.network import BlockBlastNetwork
    torch.manual_seed(9)
    base = BlockBlastNetwork().cuda()
    for m in base.modules():
        if isinstance(m, torch.nn.Dropout):
            m.p = 0.0
        if isinstance(m, torch.nn.Conv2d):                 # the reference zero-initialises biases; make them count
            torch.nn.init.normal_(m.bias, std=0.3)
    x = (torch.rand(1024, 4, 8, 8, device="cuda") < 0.4).float()

    def run(net, bf16):
        net.train()
        xin = x.contiguous(memory_format=torch.channels_last) if bf16 else x
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=bf16):
            logits, value = net.trunk(xin)
        (logits.float().pow(2).mean() + value.float().mean()).backward()
        return (logits.float().detach(), value.float().detach(), {k: (p.grad.float() if p.grad is not None else torch.zeros_like(p)) for k, p in net.named_parameters()},
                {k: b.float().clone() for k, b in net.named_buffers()})

    ref = run(copy.deepcopy(base), False)
    tor = run(copy.deepcopy(base).to(memory_format=torch.channels_last), True)
    fus_net = copy.deepcopy(base).to(memory_format=torch.channels_last).set_fused_bn(True)
    fus = run(fus_net, True)

    def rel(a, b):
        return float((a - b).norm() / (b.norm() + 1e-12))

    for i in (0, 1):
        assert rel(fus[i], ref[i]) < max(1.5 * rel(tor[i], ref[i]), 0.02), (i, rel(fus[i], ref[i]), rel(tor[i], ref[i]))
    worst = 0.0
    scale = max(float(g.norm()) for g in ref[2].values())
    for k in ref[2]:
        if float(ref[2][k].norm()) < 1e-4 * scale:
            # a conv bias in front of a BatchNorm has zero true gradient (the mean is removed):
            # what is left is rounding noise on every path, compare it in absolute terms
            assert float(fus[2][k].norm()) < max(2.0 * float(tor[2][k].norm()), 1e-3 * scale), k
            continue
        ef, et = rel(fus[2][k], ref[2][k]), rel(tor[2][k], ref[2][k])
        assert ef < max(1.5 * et, 0.03), (k, ef, et)
        worst = max(worst, ef)
    assert worst < 0.25
    for k in ref[3]:
        if k.endswith("num_batches_tracked"):
            assert float(fus[3][k]) == float(ref[3][k]) == 1.0
        else:
            assert rel(fus[3][k], ref[3][k]) < max(1.5 * rel(tor[3][k], ref[3][k]), 0.01), k
    # eval mode (deterministic evaluation) goes through the running statistics
    tor_net = copy.deepcopy(fus_net).set_fused_bn(False)
    fus_net.eval(); tor_net.eval()
    xin = x.contiguous(memory_format=torch.channels_last)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        la, _ = tor_net.trunk(xin)
        lb, _ = fus_net.trunk(xin)
    assert rel(lb.float(), la.float()) < 0.03


def test_sampling_noise_is_keyed_by_the_global_row(torch):
    """K3's Philox stream is (seed, row_offset + row, call counter): a batch sampled in two shards with their
    global offsets draws exactly what the unsharded batch draws (env shards on several GPUs / ranks), whatever
    the grid the persistent kernel runs on; a device-resident counter adds to the host one."""
    from bbgpu import capi
    g = torch.Generator(device="cuda").manual_seed(12)
    n = 3001
    logits = torch.randn(n, 192, device="cuda", generator=g)
    mask = torch.randint(-2 ** 62, 2 ** 62, (3, n), dtype=torch.int64, device="cuda", generator=g) | 1
    whole, lp = torch.empty(n, dtype=torch.int32, device="cuda"), torch.empty(n, device="cuda")
    capi.masked_sample(logits, mask, n, 5, 9, 0, whole, lp, None)
    cut = 1234
    parts, lps = torch.empty(n, dtype=torch.int32, device="cuda"), torch.empty(n, device="cuda")
    capi.masked_sample(logits[:cut].contiguous(), mask[:, :cut].contiguous(), cut, 5, 9, 0, parts[:cut], lps[:cut], None, 0)
    capi.masked_sample(logits[cut:].contiguous(), mask[:, cut:].contiguous(), n - cut, 5, 9, 0, parts[cut:], lps[cut:], None, cut)
    torch.cuda.synchronize()
    assert torch.equal(whole, parts) and torch.equal(lp, lps)
    ctr = torch.tensor([4], dtype=torch.int64, device="cuda")
    dev_ctr = torch.empty(n, dtype=torch.int32, device="cuda")
    capi.masked_sample(logits, mask, n, 5, 5, 0, dev_ctr, lp, None, 0, ctr)            # 5 + 4 == 9
    torch.cuda.synchronize()
    assert torch.equal(whole, dev_ctr)
    other = torch.empty(n, dtype=torch.int32, device="cuda")
    capi.masked_sample(logits, mask, n, 5, 9, 0, other, lp, None, 7)                   # shifted rows: different draws
    assert (other != whole).float().mean() > 0.5
