"""GPU checks of the board-symmetric policy (K7): the eight-view observation kernel (bb_unpack_obs_sym) against
K2 on host-transformed rows, the logit average (bb_sym_logits_mean) and its backward against torch formulations,
the equivariance of K1 on the device, the equivariance of the symmetrized agent, and the symmetric training and
evaluation paths end to end (rollout rows and evaluation episodes replayed through the oracles)."""
import os

import numpy as np
import pytest

import hostsym as S

pytestmark = pytest.mark.gpu

BAND = 4096
SIZES = [1, 2, 31, 33, 127, 129, 1000, 4097, 262144]


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


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


def _rows(n, rs):
    """random packed rows: any board, ids 0..36 (and a few >= 37), random used bits"""
    board = rs.randint(0, 2 ** 63, n, dtype=np.int64).astype(np.uint64) | (rs.randint(0, 2, n).astype(np.uint64) << np.uint64(63))
    ids = rs.randint(0, 37, (n, 3))
    ids[rs.rand(n, 3) < 0.02] = 40 + rs.randint(0, 200)
    used = (rs.rand(n, 3) < 0.3).astype(np.int64)
    pieces = (ids[:, 0] | (ids[:, 1] << 8) | (ids[:, 2] << 16) | (used[:, 0] << 24) | (used[:, 1] << 25) | (used[:, 2] << 26))
    return board, pieces.astype(np.uint32)


def _dev(torch, a, dtype):
    return torch.as_tensor(np.ascontiguousarray(a).view({torch.int64: np.int64, torch.int32: np.int32}[dtype])).cuda()


@pytest.mark.parametrize("with_index", [False, True])
@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
@pytest.mark.parametrize("n", SIZES)
def test_eight_views_equal_k2_on_host_transformed_rows(torch, banded, n, dtype, with_index):
    from bbgpu import capi
    dt = getattr(torch, dtype)
    rs = np.random.RandomState(n)
    m = n + 17 if with_index else n                 # source rows; the index gathers n of them
    board, pieces = _rows(m, rs)
    idx = rs.randint(0, m, n).astype(np.int64) if with_index else np.arange(n)
    b_d, p_d = _dev(torch, board, torch.int64), _dev(torch, pieces, torch.int32)
    obs = banded((8 * n, 4, 8, 8), dt)
    index = _dev(torch, idx, torch.int64) if with_index else None
    capi.unpack_obs_sym(b_d, p_d, obs, index=index, n=n)
    ref = torch.empty((n, 4, 8, 8), dtype=dt, device="cuda")
    for g in range(8):
        bg, pg = S.sym_rows(g, board[idx], pieces[idx])
        capi.unpack_obs(_dev(torch, bg, torch.int64), _dev(torch, pg, torch.int32), None, n, obs=ref, n=n)
        assert torch.equal(obs[g * n:(g + 1) * n].view(torch.int16 if dt == torch.bfloat16 else torch.int32),
                           ref.view(torch.int16 if dt == torch.bfloat16 else torch.int32)), g


def _gather_plan(torch, pieces):
    """(valid flat output positions i*192 + j, their eight view positions [8, V] as flat indices into [8n,192])"""
    from bbgpu import capi
    perm, shift = S.tables()
    cell = np.array([[S.sym_cell(g, a) for a in range(64)] for g in range(8)], np.int64)
    inb = [int(x) for x in capi.piece_table()[1]]
    n = len(pieces)
    j = np.arange(192)
    s, a = j >> 6, j & 63
    ids = (pieces[:, None].astype(np.int64) >> (8 * s)[None, :]) & 0xFF                           # [n,192]
    inb_bits = np.zeros((38, 64), bool)
    for p in range(37):
        inb_bits[p] = [(inb[p] >> k) & 1 for k in range(64)]
    valid = inb_bits[np.minimum(ids, 37), a[None, :]]
    i_idx, j_idx = np.nonzero(valid)
    idv = ids[i_idx, j_idx]
    pos = [(g * n + i_idx) * 192 + (j_idx & ~63) + cell[g][j_idx & 63] - shift[g][idv].astype(np.int64) for g in range(8)]
    return torch.as_tensor(i_idx * 192 + j_idx).cuda(), torch.as_tensor(np.stack(pos)).cuda()


@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
@pytest.mark.parametrize("n", [1, 33, 4097, 262144])
def test_logit_average_forward_and_backward(torch, banded, n, dtype):
    """forward against a float64 gather formulation within the bound of an 8-term f32 sum; backward bit for bit
    against autograd through the same formulation (scaling by 0.125 is exact, each position takes one term)."""
    from bbgpu import capi
    from bbgpu.network import SymmetryMean
    dt = getattr(torch, dtype)
    rs = np.random.RandomState(n + 1)
    _, pieces = _rows(n, rs)
    p_d = _dev(torch, pieces, torch.int32)
    logits = banded((8 * n, 192), dt)
    logits.copy_(torch.randn((8 * n, 192), device="cuda", generator=torch.Generator("cuda").manual_seed(n)) * 3)
    out = banded((n, 192), torch.float32)
    capi.sym_logits_mean(logits, p_d, out)
    flat_out, pos = _gather_plan(torch, pieces)
    L64 = logits.double().reshape(-1)
    terms = L64[pos]                                                     # [8, V]
    ref = torch.zeros(n * 192, dtype=torch.float64, device="cuda")
    ref[flat_out] = 0.125 * terms.sum(0)
    bound = 0.125 * 8 * 2.0 ** -24 * terms.abs().sum(0)
    err = (out.reshape(-1).double()[flat_out] - ref[flat_out]).abs()
    assert bool((err <= bound + 1e-30).all()), float((err - bound).max())
    untouched = torch.ones(n * 192, dtype=torch.bool, device="cuda")
    untouched[flat_out] = False
    assert not bool(out.reshape(-1)[untouched].any())
    # backward: kernel vs autograd of the torch formulation (f32 leaf, gradient cast to the logits' dtype)
    dout = torch.randn((n, 192), device="cuda", generator=torch.Generator("cuda").manual_seed(n + 7))
    grad = banded((8 * n, 192), dt)
    capi.sym_logits_mean_backward(dout.contiguous(), p_d, grad)
    leaf = logits.float().reshape(-1).clone().requires_grad_(True)
    y = torch.zeros(n * 192, dtype=torch.float32, device="cuda").index_put((flat_out,), 0.125 * leaf[pos].sum(0))
    y.backward(dout.reshape(-1))
    want = leaf.grad.view(8 * n, 192).to(dt)
    iv = torch.int16 if dt == torch.bfloat16 else torch.int32
    assert torch.equal(grad.view(iv), want.view(iv))
    # the autograd Function is the same two kernels
    lg = logits.detach().clone().requires_grad_(True)
    o2 = SymmetryMean.apply(lg, p_d)
    assert torch.equal(o2, out)
    o2.backward(dout)
    assert torch.equal(lg.grad.view(iv), grad.view(iv))


def test_k1_is_equivariant_on_the_device(torch):
    """Two env batches, one dealt from trio table T and one from T mapped through PERM by a per-env symmetry g,
    play full episodes with random legal actions and their images: every step gives the same reward bits,
    terminated flags and info words, and the transformed board, pieces and mask."""
    from bbgpu import capi
    n, L = 512, 256
    rs = np.random.RandomState(5)
    perm, _ = S.tables()
    g = rs.randint(0, 8, n).astype(np.int32)
    T = rs.randint(0, 37, (n, L, 3)).astype(np.uint8)
    Tg = perm[g[:, None, None], T]
    hA = capi.EnvHandle(n, 1, flags=capi.ENV_NO_AUTO_RESET)
    hB = capi.EnvHandle(n, 1, flags=capi.ENV_NO_AUTO_RESET)
    hA.set_trios(T)
    hB.set_trios(Tg)
    hA.reset()
    hB.reset()
    z = lambda dt, *s: torch.zeros(s, dtype=dt, device="cuda")
    oa = dict(rew=z(torch.float32, n), term=z(torch.uint8, n), mask=z(torch.int64, 3, n), info=z(torch.int32, n),
              board=z(torch.int64, n), pieces=z(torch.int32, n))
    ob = {k: torch.zeros_like(v) for k, v in oa.items()}
    hA.observe(oa["board"], oa["pieces"], oa["mask"])
    hB.observe(ob["board"], ob["pieces"], ob["mask"])
    done = np.zeros(n, bool)
    steps = 0
    while not done.all():
        ba, pa, ma = (oa[k].cpu().numpy().view(t) for k, t in (("board", np.uint64), ("pieces", np.uint32), ("mask", np.uint64)))
        bb, pb, mb = (ob[k].cpu().numpy().view(t) for k, t in (("board", np.uint64), ("pieces", np.uint32), ("mask", np.uint64)))
        bt, pt = S.sym_rows(g, ba, pa)
        assert np.array_equal(bb, bt) and np.array_equal(pb, pt), steps
        assert np.array_equal(mb, S.sym_mask_rows(g, pa, ma)), steps
        act = np.zeros(n, np.int32)
        for i in np.flatnonzero(~done):
            legal = [k * 64 + a for k in range(3) for a in range(64) if (int(ma[k, i]) >> a) & 1]
            act[i] = legal[rs.randint(len(legal))]
        act_g = np.where(done, 0, S.sym_action_rows(g, pa, act))
        for h, o, a in ((hA, oa, act), (hB, ob, act_g)):
            h.step(torch.as_tensor(a).cuda(), o["rew"], o["term"], o["mask"], info_out=o["info"], board_out=o["board"],
                   pieces_out=o["pieces"])
        live = ~done
        assert np.array_equal(oa["rew"].cpu().numpy().view(np.uint32)[live], ob["rew"].cpu().numpy().view(np.uint32)[live])
        assert np.array_equal(oa["term"].cpu().numpy()[live], ob["term"].cpu().numpy()[live])
        assert np.array_equal(oa["info"].cpu().numpy()[live], ob["info"].cpu().numpy()[live])
        assert not (oa["info"].cpu().numpy()[live] & 1).any()          # every action legal
        done |= oa["term"].cpu().numpy().astype(bool)
        steps += 1
    sa, sb = hA.get_state(), hB.get_state()
    for f in ("score", "moves", "lines_total", "max_streak", "blocks_total", "draw_ctr"):
        assert np.array_equal(sa[f], sb[f]), f
    assert steps > 10
    hA.close()
    hB.close()


def _midgame_obs(torch, n, seed, steps):
    """packed observations of n envs after up to ``steps`` random moves (auto-reset keeps them live)"""
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


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_symmetrized_agent_is_equivariant_in_eval_mode(torch, precision):
    from bbgpu import capi
    from bbgpu.ppo import PPOAgent, PPOConfig
    torch.manual_seed(3)
    agent = PPOAgent(PPOConfig(precision=precision, symmetrize=True), seed=1)
    agent.eval()
    n = 1024
    board, pieces, mask = _midgame_obs(torch, n, 21, 9)
    rs = np.random.RandomState(8)
    g = rs.randint(0, 8, n).astype(np.int32)
    pa = pieces.cpu().numpy().view(np.uint32)
    bg, pg = S.sym_rows(g, board.cpu().numpy().view(np.uint64), pa)
    mg = S.sym_mask_rows(g, pa, mask.cpu().numpy().view(np.uint64))
    obs = {"board": board, "pieces": pieces, "mask": mask}
    obs_g = {"board": _dev(torch, bg, torch.int64), "pieces": _dev(torch, pg, torch.int32), "mask": _dev(torch, mg, torch.int64)}
    with torch.no_grad():
        la, va, _ = agent._policy(obs)
        lb, vb, _ = agent._policy(obs_g)
    tol = 1e-4 if precision == "fp32" else 2e-3
    assert torch.allclose(va, vb, rtol=tol, atol=tol), float((va - vb).abs().max())
    # log-probs of corresponding actions (K3 mode 2)
    ma = mask.cpu().numpy().view(np.uint64)
    act = np.zeros(n, np.int32)
    for i in range(n):
        legal = [k * 64 + a for k in range(3) for a in range(64) if (int(ma[k, i]) >> a) & 1]
        act[i] = legal[rs.randint(len(legal))] if legal else 0
    has = ma.any(axis=0)
    act_g = np.where(has, S.sym_action_rows(g, pa, act), 0).astype(np.int32)
    lp_a = torch.empty(n, device="cuda")
    lp_b = torch.empty(n, device="cuda")
    capi.masked_sample(la, mask, n, 0, 0, 2, torch.as_tensor(act).cuda(), lp_a)
    capi.masked_sample(lb, obs_g["mask"], n, 0, 0, 2, torch.as_tensor(act_g).cuda(), lp_b)
    hv = torch.as_tensor(has).cuda()
    assert torch.allclose(lp_a[hv], lp_b[hv], rtol=tol, atol=10 * tol), float((lp_a - lp_b)[hv].abs().max())
    # argmax maps wherever the top-two margin of the masked logits exceeds the tolerance
    am_a = torch.empty(n, dtype=torch.int32, device="cuda")
    am_b = torch.empty(n, dtype=torch.int32, device="cuda")
    capi.masked_sample(la, mask, n, 0, 0, 1, am_a, torch.empty(n, device="cuda"))
    capi.masked_sample(lb, obs_g["mask"], n, 0, 0, 1, am_b, torch.empty(n, device="cuda"))
    dense = torch.zeros((n, 192), dtype=torch.uint8, device="cuda")
    capi.unpack_obs(None, None, mask, n, mask_dense=dense, n=n)
    top2 = la.masked_fill(dense == 0, float("-inf")).topk(2, dim=1).values
    margin = (top2[:, 0] - top2[:, 1]).cpu().numpy()
    clear = has & (margin > 10 * tol)
    mapped = S.sym_action_rows(g, pa, am_a.cpu().numpy())
    assert clear.sum() > n // 2
    assert np.array_equal(mapped[clear], am_b.cpu().numpy()[clear])


def _runner_rollouts(torch, use_graph, n, T, seed, rollouts):
    from bbgpu.ppo import PPOAgent, PPOConfig
    from bbgpu.rollout import RolloutBuffer
    from bbgpu.train import RolloutRunner
    from bbgpu.vec_env import VectorizedBlockBlastEnv
    torch.manual_seed(0)
    agent = PPOAgent(PPOConfig(precision="fp32", symmetrize=True), seed=seed)
    agent.train()
    venv = VectorizedBlockBlastEnv(n, seed=seed, output="packed")
    buf = RolloutBuffer(T, n)
    runner = RolloutRunner(venv, agent, buf, use_graph=use_graph)
    assert runner.x_buf.shape[0] == 8 * n
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


def test_symmetric_rollout_eager_equals_graph_and_replays_through_the_oracle(torch):
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


def test_short_symmetric_training_and_checkpoint_round_trip(torch, tmp_path):
    from bbgpu.ppo import PPOAgent, PPOConfig
    from bbgpu.train import train
    cfg = {"training": {"num_envs": 256, "batch_size": 1024, "rollout_steps": 8, "total_timesteps": 256 * 8 * 3},
           "ppo": {"num_epochs": 2}, "logging": {"log_interval": 1, "save_interval": 100, "tensorboard": False},
           "paths": {"checkpoint_dir": str(tmp_path / "ck"), "log_dir": str(tmp_path / "logs")},
           "b200": {"precision": "bf16", "symmetrize": True}}
    hist = train(cfg, seed=3)
    assert len(hist) == 3 and all(np.isfinite(h["policy_loss"]) and h["entropy"] > 0.1 for h in hist)
    ck = torch.load(str(tmp_path / "ck" / "final.pt"), weights_only=True)
    assert set(ck) == {"network_state_dict", "optimizer_state_dict", "config", "b200_state"}
    assert "symmetrize" not in ck["config"] and "precision" not in ck["config"] and ck["b200_state"]["symmetrize"] is True
    agent = PPOAgent(PPOConfig())
    assert agent.config.symmetrize is False
    agent.load(str(tmp_path / "ck" / "final.pt"))
    assert agent.config.symmetrize is True
    agent.save(str(tmp_path / "again.pt"))
    plain = PPOAgent(PPOConfig(symmetrize=True))
    plain.config.symmetrize = False
    plain.save(str(tmp_path / "plain.pt"))
    agent.load(str(tmp_path / "plain.pt"))
    assert agent.config.symmetrize is False
    agent.load(str(tmp_path / "again.pt"))
    assert agent.config.symmetrize is True


@pytest.mark.parametrize("lookahead", [0, 1])
def test_symmetric_evaluation_replays_through_the_oracle(torch, lookahead):
    from bbgpu import philox
    from bbgpu.evaluate import evaluate
    from bbgpu.ppo import PPOAgent
    from oracle import bb_oracle as O
    torch.manual_seed(5)
    agent = PPOAgent()
    n, seed = 32, 17
    res = evaluate(agent, num_episodes=n, seed=seed, return_actions=True, lookahead=lookahead, symmetrize=True)
    assert agent.config.symmetrize is False and res["finished"] == n
    # the first moves are the eight-view policy's (recomputed on the same initial states), not the plain one's
    from bbgpu import capi
    from bbgpu.evaluate import lookahead_actions
    first = {}
    agent.eval()
    for sym in (True, False):
        agent.config.symmetrize = sym
        h = capi.EnvHandle(n, seed, 0, None, capi.ENV_NO_AUTO_RESET)
        if lookahead:
            act, _, _ = lookahead_actions(agent, h, n, 0, lookahead)
        else:
            board = torch.zeros(n, dtype=torch.int64, device="cuda")
            pieces = torch.zeros(n, dtype=torch.int32, device="cuda")
            mask = torch.zeros((3, n), dtype=torch.int64, device="cuda")
            h.observe(board, pieces, mask)
            act, _, _ = agent.act({"board": board, "pieces": pieces, "mask": mask}, deterministic=True)
        first[sym] = act.cpu().numpy()
        h.close()
    agent.config.symmetrize = False
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
