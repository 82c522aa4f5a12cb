"""GPU checks of the canonical-frame policy (K7c, PPOConfig.canonical_frame): the canonical-view kernel
(bb_sym_canonical) against its host build and its planes against the eight-view kernel, the logit map
(bb_sym_logits_canonical) and its backward against torch formulations, the exact invariance of the agent, one
update against an independent restatement, and the training and evaluation paths end to end (rollout rows and
evaluation episodes replayed through the oracles)."""
import numpy as np
import pytest

import hostcanon as K
import hostsym as S

pytestmark = pytest.mark.gpu

BAND = 4096
SIZES = [1, 2, 31, 33, 127, 129, 1000, 4097, 262144]


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


@pytest.fixture(autouse=True)
def _cudnn_flags(torch):
    """A bf16 PPOAgent turns on cudnn.benchmark for the whole process; restore the flags after every test so that
    the tests that run later see the convolution algorithms they would see without this file."""
    flags = torch.backends.cudnn.benchmark, torch.backends.cudnn.deterministic
    yield
    torch.backends.cudnn.benchmark, torch.backends.cudnn.deterministic = flags


@pytest.fixture
def banded(torch):
    """Allocator of device tensors with a 4 KB band of a known byte pattern on both sides; the bands are
    checked when the test ends."""
    made = []

    def alloc(shape, dtype):
        n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
        buf = torch.full((n + 2 * BAND,), 0xA5, dtype=torch.uint8, device="cuda")
        made.append(buf)
        return buf[BAND:BAND + n].view(dtype).view(*shape)

    yield alloc
    torch.cuda.synchronize()
    for buf in made:
        assert bool((buf[:BAND] == 0xA5).all()) and bool((buf[-BAND:] == 0xA5).all()), "guard band overwritten"


def _dev(torch, a, dtype):
    return torch.as_tensor(np.ascontiguousarray(a).view({torch.int64: np.int64, torch.int32: np.int32,
                                                         torch.uint8: np.uint8}[dtype])).cuda()


def _mixed_rows(n, rs):
    """random rows, with up to 2,000 rows of every stabiliser order spread through them"""
    board, pieces = K.random_rows(n, rs)
    k = min(n, 2000)
    at = rs.choice(n, k, replace=False)
    parts = [K.symmetric_rows(k // len(K.SUBGROUPS) + 1, h, rs) for h in K.SUBGROUPS]
    board[at] = np.concatenate([b for b, _ in parts])[:k]
    pieces[at] = np.concatenate([p for _, p in parts])[:k]
    return board, pieces


@pytest.mark.parametrize("with_index", [False, True])
@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
@pytest.mark.parametrize("n", SIZES)
def test_canonical_kernel_equals_host_and_its_planes_equal_the_view_planes(torch, banded, n, dtype, with_index):
    from bbgpu import capi
    dt = getattr(torch, dtype)
    rs = np.random.RandomState(n + 3)
    m = n + 17 if with_index else n
    board, pieces = _mixed_rows(m, rs)
    idx = rs.randint(0, m, n).astype(np.int64) if with_index else np.arange(n)
    b_d, p_d = _dev(torch, board, torch.int64), _dev(torch, pieces, torch.int32)
    index = _dev(torch, idx, torch.int64) if with_index else None
    cb, cp, v = banded((n,), torch.int64), banded((n,), torch.int32), banded((n,), torch.uint8)
    capi.sym_canonical(b_d, p_d, cb, cp, v, index=index, n=n)
    hb, hp, hv = K.canonical(board[idx], pieces[idx])
    assert np.array_equal(cb.cpu().numpy().view(np.uint64), hb)
    assert np.array_equal(cp.cpu().numpy().view(np.uint32), hp)
    assert np.array_equal(v.cpu().numpy(), hv)
    # K2 on the canonical rows = the row of the eight-view observation of one view in M
    obs = banded((n, 4, 8, 8), dt)
    capi.unpack_obs(cb, cp, None, n, obs=obs, n=n)
    views = torch.empty((8 * n, 4, 8, 8), dtype=dt, device="cuda")
    capi.unpack_obs_sym(b_d, p_d, views, index=index, n=n)
    g0 = torch.as_tensor(np.array([(int(x) & -int(x)).bit_length() - 1 for x in hv], np.int64)).cuda()
    iv = torch.int16 if dt == torch.bfloat16 else torch.int32
    want = views[g0 * n + torch.arange(n, device="cuda")]
    assert torch.equal(obs.view(iv), want.view(iv))


def _map_plan(torch, pieces, views):
    """(valid flat output positions i*192 + j [V], canonical positions [8, V] of each view g as flat indices into
    [n,192], view membership [8, V] as float64, |M| [V])"""
    from bbgpu import capi
    _, shift = S.tables()
    cell = np.array([[S.sym_cell(g, a) for a in range(64)] for g in range(8)], np.int64)
    inb = [int(x) for x in capi.piece_table()[1]]
    j = np.arange(192)
    s, a = j >> 6, j & 63
    ids = (pieces[:, None].astype(np.int64) >> (8 * s)[None, :]) & 0xFF
    inb_bits = np.zeros((38, 64), bool)
    for p in range(37):
        inb_bits[p] = [(inb[p] >> k) & 1 for k in range(64)]
    valid = inb_bits[np.minimum(ids, 37), a[None, :]]
    i_idx, j_idx = np.nonzero(valid)
    idv = ids[i_idx, j_idx]
    pos = np.stack([i_idx * 192 + (j_idx & ~63) + cell[g][j_idx & 63] - shift[g][idv].astype(np.int64) for g in range(8)])
    member = np.stack([(views[i_idx] >> g) & 1 for g in range(8)]).astype(np.float64)
    cnt = member.sum(0)
    cuda = lambda x: torch.as_tensor(x).cuda()
    return cuda(i_idx * 192 + j_idx), cuda(pos), cuda(member), cuda(cnt)


def _torch_map(torch, flat, logits, plan):
    """the map as a torch gather: out[i, j] = sum_{g in M} L[pos_g] / |M|, 0 at invalid positions"""
    flat_out, pos, member, cnt = plan
    n = logits.shape[0]
    lv = logits.reshape(-1)
    y = (lv[pos] * member.to(lv.dtype)).sum(0) / cnt.to(lv.dtype)
    return torch.zeros(n * 192, dtype=lv.dtype, device="cuda").index_put((flat_out,), y).view(n, 192)


@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
@pytest.mark.parametrize("n", [1, 33, 4097, 262144])
def test_logit_map_forward_and_backward(torch, banded, n, dtype):
    from bbgpu import capi
    from bbgpu.network import CanonicalFrame
    dt = getattr(torch, dtype)
    rs = np.random.RandomState(n + 11)
    board, pieces = _mixed_rows(n, rs)
    _, _, views = K.canonical(board, pieces)
    p_d, v_d = _dev(torch, pieces, torch.int32), _dev(torch, views, torch.uint8)
    logits = banded((n, 192), dt)
    logits.copy_(torch.randn((n, 192), device="cuda", generator=torch.Generator("cuda").manual_seed(n)) * 3)
    out = banded((n, 192), torch.float32)
    capi.sym_logits_canonical(logits, p_d, v_d, out)
    plan = _map_plan(torch, pieces, views)
    flat_out, pos, member, cnt = plan
    ref = _torch_map(torch, None, logits.double(), plan).reshape(-1)
    terms = logits.double().reshape(-1)[pos].abs() * member
    bound = 8 * 2.0 ** -24 * terms.sum(0) / cnt
    got = out.reshape(-1).double()
    err = (got[flat_out] - ref[flat_out]).abs()
    assert bool((err <= bound + 1e-30).all()), float((err - bound).max())
    one = cnt == 1
    assert torch.equal(got[flat_out][one], ref[flat_out][one])           # one term: exact
    untouched = torch.ones(n * 192, dtype=torch.bool, device="cuda")
    untouched[flat_out] = False
    assert not bool(got[untouched].any())
    # backward: kernel vs autograd of the torch formulation (f32 leaf, gradient cast to the logits' dtype)
    dout = torch.randn((n, 192), device="cuda", generator=torch.Generator("cuda").manual_seed(n + 7))
    grad = banded((n, 192), dt)
    capi.sym_logits_canonical_backward(dout.contiguous(), p_d, v_d, grad)
    leaf = logits.float().clone().requires_grad_(True)
    _torch_map(torch, None, leaf, plan).backward(dout)
    want = leaf.grad.to(dt)
    iv = torch.int16 if dt == torch.bfloat16 else torch.int32
    rows_one = torch.as_tensor(np.array([bin(int(x)).count("1") == 1 for x in views])).cuda()
    assert torch.equal(grad[rows_one].view(iv), want[rows_one].view(iv))  # |M| = 1: a permutation, exact
    if bool((~rows_one).any()):                                           # |M| > 1: collisions, within the sum bound
        gs, ws = grad[~rows_one].float(), want[~rows_one].float()
        tol = 8 * 2.0 ** -24 * dout.abs().max() + (2.0 ** -8 if dt == torch.bfloat16 else 0.0) * ws.abs()
        assert bool(((gs - ws).abs() <= tol + 1e-30).all()), float((gs - ws).abs().max())
    # zero where no output position reaches
    reach = torch.zeros(n * 192, dtype=torch.bool, device="cuda")
    reach[pos[member.bool()]] = True
    assert not bool(grad.reshape(-1)[~reach].float().any())
    # repeated runs are bitwise identical
    out2, grad2 = torch.empty_like(out), torch.empty_like(grad)
    capi.sym_logits_canonical(logits, p_d, v_d, out2)
    capi.sym_logits_canonical_backward(dout.contiguous(), p_d, v_d, grad2)
    assert torch.equal(out2, out) and torch.equal(grad2.view(iv), grad.view(iv))
    # the autograd Function is the same two kernels
    lg = logits.detach().clone().requires_grad_(True)
    o2 = CanonicalFrame.apply(lg, p_d, v_d)
    assert torch.equal(o2, out)
    o2.backward(dout)
    assert torch.equal(lg.grad.view(iv), grad.view(iv))


def _midgame_obs(torch, n, seed, steps):
    from bbgpu import capi
    h = capi.EnvHandle(n, seed)
    h.step_random(steps)
    board = torch.zeros(n, dtype=torch.int64, device="cuda")
    pieces = torch.zeros(n, dtype=torch.int32, device="cuda")
    mask = torch.zeros((3, n), dtype=torch.int64, device="cuda")
    h.observe(board, pieces, mask)
    torch.cuda.synchronize()
    h.close()
    return board, pieces, mask


@pytest.mark.parametrize("mode", ["eval", "train"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_canonical_agent_is_exactly_invariant(torch, precision, mode):
    """values bit for bit; logits at mapped positions bit for bit where |M| = 1, within the sum bound elsewhere
    (the same terms in another order).  Train mode: BatchNorm sees identical rows, dropout is re-seeded."""
    from bbgpu.ppo import PPOAgent, PPOConfig
    torch.manual_seed(3)
    agent = PPOAgent(PPOConfig(precision=precision, canonical_frame=True), seed=1)
    agent.eval() if mode == "eval" else agent.train()
    n = 1024
    board, pieces, mask = _midgame_obs(torch, n, 21, 9)
    rs = np.random.RandomState(8)
    g = rs.randint(0, 8, n).astype(np.int32)
    pa = pieces.cpu().numpy().view(np.uint32)
    bg, pg = S.sym_rows(g, board.cpu().numpy().view(np.uint64), pa)
    # a few states with a non-trivial stabiliser: empty boards with the fully symmetric trio
    pa = pa.copy()
    bnp = board.cpu().numpy().view(np.uint64).copy()
    bnp[:8], pa[:8] = 0, K.pack([[0, 17, 36]] * 8, [[0, 0, 0]] * 8)
    bg[:8], pg[:8] = bnp[:8], pa[:8]
    obs = {"board": _dev(torch, bnp, torch.int64), "pieces": _dev(torch, pa, torch.int32), "mask": mask}
    obs_g = {"board": _dev(torch, bg, torch.int64), "pieces": _dev(torch, pg, torch.int32), "mask": mask}
    det = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        with torch.no_grad():
            torch.manual_seed(99)
            la, va, _ = agent._policy(obs)
            torch.manual_seed(99)
            lb, vb, _ = agent._policy(obs_g)
    finally:
        torch.backends.cudnn.deterministic = det
    assert torch.equal(va, vb)
    _, _, views = K.canonical(bnp, pa)
    assert (views[:8] == 0xFF).all()
    flat_out, pos, _, cnt = _map_plan(torch, pa, np.ones(n, np.uint8))   # pos[g]: image of j under view g
    gi = torch.as_tensor(g.astype(np.int64)).cuda()[flat_out // 192]
    img = pos.gather(0, gi[None])[0]
    a, b = la.reshape(-1)[flat_out], lb.reshape(-1)[img]
    size = torch.as_tensor(np.array([bin(int(x)).count("1") for x in views])).cuda()[flat_out // 192]
    one = size == 1
    assert bool(one.any()) and bool((~one).any())
    assert torch.equal(a[one], b[one])
    tol = 8 * 2.0 ** -24 * a[~one].abs() * 8 + 1e-6
    assert bool(((a[~one] - b[~one]).abs() <= tol).all())


def test_minibatch_step_metrics_match_independent_computation(torch):
    """One epoch, one minibatch = the whole buffer, eval mode: the metrics of PPOAgent.update with canonical_frame
    equal ppo.py:372-406 on the network's logits of host-canonicalised rows mapped back with a torch gather."""
    from bbgpu import capi
    from bbgpu.ppo import PPOAgent, PPOConfig
    from bbgpu.rollout import RolloutBuffer
    from bbgpu.train import RolloutRunner
    from bbgpu.vec_env import VectorizedBlockBlastEnv
    from bbgpu import vec_env as VE
    from oracle import bb_oracle as O
    torch.manual_seed(0)
    T, N = 8, 64
    agent = PPOAgent(PPOConfig(num_epochs=1, batch_size=T * N, learning_rate=1e-3, canonical_frame=True))
    agent.eval()
    venv = VectorizedBlockBlastEnv(N, seed=9, output="packed")
    venv.reset()
    buf = RolloutBuffer(T, N)
    last = RolloutRunner(venv, agent, buf, use_graph=False).run()
    assert (buf.rewards > -5).all()
    bo = buf.boards[:T].reshape(-1).cpu().numpy().view(np.uint64)
    po = buf.pieces[:T].reshape(-1).cpu().numpy().view(np.uint32)
    cb, cp, views = K.canonical(bo, po)
    x = torch.empty((T * N, 4, 8, 8), dtype=torch.float32, device="cuda")
    capi.unpack_obs(_dev(torch, cb, torch.int64), _dev(torch, cp, torch.int32), None, T * N, obs=x, n=T * N)
    with torch.no_grad():
        logits, values = agent.network.trunk(x)
    mapped = _torch_map(torch, None, logits.double(), _map_plan(torch, po, views)).cpu().numpy()
    g = buf.gather(torch.arange(T * N, device="cuda"), None)
    dense = VE.expand_mask(g["mask"].cpu().numpy().view(np.uint64)).astype(np.float32)
    adv, ret = O.gae(buf.rewards.cpu().numpy(), buf.values.cpu().numpy(), buf.dones.cpu().numpy(), last.cpu().numpy(), 0.99, 0.95)
    a_n = O.normalize_advantages(adv)
    acts = buf.actions.view(-1).cpu().numpy()
    _, new_lp, ent = O.masked_policy_terms(mapped, dense, acts)
    old_lp = buf.log_probs.view(-1).cpu().numpy()
    np.testing.assert_allclose(new_lp, old_lp, rtol=1e-4, atol=1e-5)
    ratio = np.exp(new_lp - old_lp)
    pol = -np.minimum(ratio * a_n, np.clip(ratio, 0.8, 1.2) * a_n).mean()
    vl = ((values.cpu().numpy() - ret.reshape(-1)) ** 2).mean()
    np.testing.assert_allclose(values.cpu().numpy(), buf.values.view(-1).cpu().numpy(), rtol=1e-4, atol=1e-5)
    before = [p.detach().clone() for p in agent.network.parameters()]
    m = agent.update(buf, last)
    assert abs(m["policy_loss"] - pol) < 1e-4 and abs(m["value_loss"] - vl) < 1e-3 * max(1.0, vl)
    assert abs(m["entropy"] - ent.mean()) < 1e-4
    assert abs(m["total_loss"] - (pol + 0.5 * vl - 0.01 * ent.mean())) < 1e-3 * max(1.0, vl)
    assert m["clip_fraction"] < 1e-3 and abs(m["approx_kl"]) < 1e-4
    assert any(not torch.equal(a, b) for a, b in zip(before, agent.network.parameters()))
    venv.close()


def _runner_rollouts(torch, use_graph, n, T, seed, rollouts):
    from bbgpu.ppo import PPOAgent, PPOConfig
    from bbgpu.rollout import RolloutBuffer
    from bbgpu.train import RolloutRunner
    from bbgpu.vec_env import VectorizedBlockBlastEnv
    torch.manual_seed(0)
    agent = PPOAgent(PPOConfig(precision="fp32", canonical_frame=True), seed=seed)
    agent.train()
    venv = VectorizedBlockBlastEnv(n, seed=seed, output="packed")
    buf = RolloutBuffer(T, n)
    runner = RolloutRunner(venv, agent, buf, use_graph=use_graph)
    assert runner.x_buf.shape[0] == n and runner.canon is not None
    rows = []
    for _ in range(rollouts):
        lv = runner.run()
        torch.cuda.synchronize()
        rows.append({k: getattr(buf, k).clone() for k in ("boards", "pieces", "action_masks", "actions", "log_probs",
                                                          "rewards", "terminated", "values")})
        rows[-1]["last_values"] = lv.clone()
    m = agent.update(buf, lv, use_graph=use_graph)
    m2 = agent.update(buf, lv, use_graph=use_graph)
    venv.close()
    return rows, (m, m2)


def test_canonical_rollout_eager_equals_graph_and_replays_through_the_oracle(torch):
    from bbgpu import philox
    from oracle import bb_oracle_c as OC
    n, T, seed = 64, 16, 13
    bench, det = torch.backends.cudnn.benchmark, torch.backends.cudnn.deterministic
    torch.backends.cudnn.benchmark, torch.backends.cudnn.deterministic = False, True
    try:
        eager, me = _runner_rollouts(torch, False, n, T, seed, 3)
        graph, mg = _runner_rollouts(torch, True, n, T, seed, 3)
    finally:
        torch.backends.cudnn.benchmark, torch.backends.cudnn.deterministic = bench, det
    for it in range(3):
        for k in eager[it]:
            assert torch.equal(eager[it][k], graph[it][k]), (it, k)
    for m in me + mg:
        assert all(np.isfinite(v) for v in m.values()) and m["entropy"] > 0.1
    ora = OC.CVecEnv(philox.candidate_trios(seed, np.arange(n), 2048))
    for it in range(3):
        r = {k: v.cpu().numpy() for k, v in graph[it].items()}
        boards, masks = r["boards"].view(np.uint64), r["action_masks"].view(np.uint64)
        pieces = r["pieces"].view(np.uint8).reshape(T + 1, n, 4)
        b0, p0, m0 = ora.export()
        assert np.array_equal(boards[0], b0) and np.array_equal(pieces[0], p0) and np.array_equal(masks[0].T, m0)
        for t in range(T):
            a = r["actions"][t]
            assert ((masks[t][a // 64, np.arange(n)] >> (a % 64).astype(np.uint64)) & np.uint64(1)).all(), (it, t)
            oo = ora.step(a)
            assert not oo["invalid"].any()
            assert np.array_equal(oo["rewards"].view(np.uint32), r["rewards"][t].view(np.uint32)), (it, t)
            assert np.array_equal(oo["terminated"], r["terminated"][t]), (it, t)
            assert np.array_equal(oo["mask"], masks[t + 1].T), (it, t)
            assert np.array_equal(oo["board"], boards[t + 1]) and np.array_equal(oo["pieces"], pieces[t + 1]), (it, t)


def test_short_canonical_training_and_checkpoint_round_trip(torch, tmp_path):
    from bbgpu.ppo import PPOAgent, PPOConfig
    from bbgpu.train import train
    cfg = {"training": {"num_envs": 256, "batch_size": 1024, "rollout_steps": 8, "total_timesteps": 256 * 8 * 3},
           "ppo": {"num_epochs": 2}, "logging": {"log_interval": 1, "save_interval": 100, "tensorboard": False},
           "paths": {"checkpoint_dir": str(tmp_path / "ck"), "log_dir": str(tmp_path / "logs")},
           "b200": {"precision": "bf16", "canonical_frame": True}}
    hist = train(cfg, seed=3)
    assert len(hist) == 3 and all(np.isfinite(h["policy_loss"]) and h["entropy"] > 0.1 for h in hist)
    ck = torch.load(str(tmp_path / "ck" / "final.pt"), weights_only=True)
    assert set(ck) == {"network_state_dict", "optimizer_state_dict", "config", "b200_state"}
    assert "canonical_frame" not in ck["config"] and "symmetrize" not in ck["config"]
    assert ck["b200_state"]["canonical_frame"] is True and ck["b200_state"]["symmetrize"] is False
    PPOConfig(**ck["config"])                                    # the reference's constructor accepts the config
    agent = PPOAgent(PPOConfig())
    agent.load(str(tmp_path / "ck" / "final.pt"))
    assert agent.config.canonical_frame is True and agent.config.symmetrize is False
    agent.save(str(tmp_path / "again.pt"))
    old = {**ck, "b200_state": {k: v for k, v in ck["b200_state"].items() if k != "canonical_frame"}}
    torch.save(old, str(tmp_path / "old.pt"))                   # written before the flag existed
    agent.load(str(tmp_path / "old.pt"))
    assert agent.config.canonical_frame is False
    agent.load(str(tmp_path / "again.pt"))
    assert agent.config.canonical_frame is True
    with pytest.raises(ValueError):
        PPOConfig(symmetrize=True, canonical_frame=True)
    with pytest.raises(ValueError):
        train({**cfg, "b200": {"symmetrize": True, "canonical_frame": True}}, seed=3)
    # --resume: the config's policy form wins over the checkpoint's
    cfg2 = {**cfg, "training": {**cfg["training"], "total_timesteps": 256 * 8 * 4}, "b200": {"precision": "bf16", "symmetrize": True}}
    hist = train(cfg2, resume_path=str(tmp_path / "ck" / "final.pt"), seed=3, max_updates=1)
    ck2 = torch.load(str(tmp_path / "ck" / "final.pt"), weights_only=True)
    assert ck2["b200_state"]["symmetrize"] is True and ck2["b200_state"]["canonical_frame"] is False


@pytest.mark.parametrize("lookahead", [0, 1])
def test_canonical_evaluation_replays_through_the_oracle(torch, lookahead):
    from bbgpu import capi, philox
    from bbgpu.evaluate import evaluate, lookahead_actions
    from bbgpu.ppo import PPOAgent
    from oracle import bb_oracle as O
    torch.manual_seed(5)
    agent = PPOAgent()
    n, seed = 32, 17
    res = evaluate(agent, num_episodes=n, seed=seed, return_actions=True, lookahead=lookahead, canonical_frame=True)
    assert agent.config.canonical_frame is False and agent.config.symmetrize is False and res["finished"] == n
    with pytest.raises(ValueError):
        evaluate(agent, num_episodes=2, symmetrize=True, canonical_frame=True)
    # the first moves are the canonical policy's (recomputed on the same initial states), not the plain one's
    first = {}
    agent.eval()
    for canon in (True, False):
        agent.config.canonical_frame = canon
        h = capi.EnvHandle(n, seed, 0, None, capi.ENV_NO_AUTO_RESET)
        if lookahead:
            act, _, _ = lookahead_actions(agent, h, n, 0, lookahead)
        else:
            board = torch.zeros(n, dtype=torch.int64, device="cuda")
            pieces = torch.zeros(n, dtype=torch.int32, device="cuda")
            mask = torch.zeros((3, n), dtype=torch.int64, device="cuda")
            h.observe(board, pieces, mask)
            act, _, _ = agent.act({"board": board, "pieces": pieces, "mask": mask}, deterministic=True)
        first[canon] = act.cpu().numpy()
        h.close()
    agent.config.canonical_frame = False
    agent.train()
    assert np.array_equal(res["actions"][0], first[True])
    assert not np.array_equal(first[True], first[False])
    streams = philox.candidate_trios(seed, np.arange(n), 1024)
    for i in range(n):
        it = iter(streams[i])
        env = O.Env(draw=lambda it=it: next(it))
        total, t, term, info = 0.0, 0, False, None
        while not term:
            _, r, term, _, info = env.step(int(res["actions"][t, i]))
            assert not info["invalid_action"], (i, t)
            total += float(np.float32(r))
            t += 1
        assert info["score"] == res["scores"][i] and info["moves"] == res["lengths"][i] == t
        assert info["lines_cleared"] == res["lines"][i] and info["max_combo"] == res["max_combos"][i]
        assert abs(total - res["rewards_per_episode"][i]) < 1e-4 * max(1.0, abs(total))


def test_act_chunks_states(torch):
    """chunked and whole-batch evaluation agree up to the CNN's batch-size-dependent rounding (eval mode)"""
    from bbgpu.ppo import PPOAgent, PPOConfig
    torch.manual_seed(4)
    agent = PPOAgent(PPOConfig(canonical_frame=True))
    agent.eval()
    board, pieces, mask = _midgame_obs(torch, 300, 2, 5)
    obs = {"board": board, "pieces": pieces, "mask": mask}
    with torch.no_grad():
        l1, v1, _ = agent._policy(obs)
        l2, v2, _ = agent._policy(obs, chunk=64)
    assert l1.shape == l2.shape == (300, 192) and v1.shape == v2.shape == (300,)
    assert torch.allclose(l1, l2, atol=2e-3) and torch.allclose(v1, v2, atol=2e-3)
    a, _, _ = agent.act(obs, deterministic=True, chunk=64)
    dense = torch.zeros((300, 192), dtype=torch.uint8, device="cuda")
    from bbgpu import capi
    capi.unpack_obs(None, None, mask, 300, mask_dense=dense, n=300)
    assert bool(dense.gather(1, a.long()[:, None]).all())
