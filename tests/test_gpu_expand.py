"""bb_env_expand on the GPU: every item against the host build of the same rules (bbx_expand, which
test_expand_host.py pins to the Python oracle), non-deal items against K1 itself, the no-state-change
and determinism contract, capacity handling with guard bands, and the look-ahead evaluation policy
built on it (decision rule and oracle replay)."""
import copy

import numpy as np
import pytest

import hostexpand as HX

pytestmark = pytest.mark.gpu
BAND = 4096
FIELDS = HX.EXPAND_FIELDS
NP_VIEW = {"action": np.int32, "reward": np.float32, "terminated": np.uint8, "info": np.uint32,
           "board": np.uint64, "pieces": np.uint32}


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


class Arena:
    """Every buffer of a call carved out of one device arena with a 4 KB band of a known byte pattern
    on both sides (the scheme of test_gpu_guard_bands.py); check() fails if a band was written."""

    def __init__(self, torch, nbytes=1 << 26):
        self.t = torch
        self.buf = torch.full((nbytes,), 0xA5, dtype=torch.uint8, device="cuda")
        self.off = BAND
        self.spans = []

    def alloc(self, shape, dtype):
        n = int(np.prod(shape)) * self.t.empty((), dtype=dtype).element_size()
        start = (self.off + 255) // 256 * 256
        self.off = start + n + BAND
        assert self.off < self.buf.numel()
        self.spans.append((start, n))
        return self.buf[start:start + n].view(dtype).view(*shape)

    def check(self):
        self.t.cuda.synchronize()
        host = self.buf[:self.off].cpu().numpy()
        keep = np.ones(self.off, bool)
        for s, n in self.spans:
            keep[s:s + n] = False
        bad = np.flatnonzero(keep & (host != 0xA5))
        assert bad.size == 0, "guard band overwritten at arena offsets %s" % bad[:8]


def _host_view(ex):
    out = {k: v.cpu().numpy() for k, v in ex.items()}
    for k, dt in NP_VIEW.items():
        out[k] = out[k].view(dt)
    out["mask"] = out["mask"].view(np.uint64)
    return out


def _midgame(torch, n, seed, max_steps=60, rseed=0, env_offset=0):
    """n envs (BB_ENV_NO_AUTO_RESET) after 0..max_steps random valid moves each (a finished env stays
    GAME_OVER); moves come from bb_env_sample_valid_actions, envs past their step budget get -1 (a no-op)."""
    from bbgpu import capi
    h = capi.EnvHandle(n, seed, env_offset, None, capi.ENV_NO_AUTO_RESET)
    g = torch.Generator(device="cuda").manual_seed(rseed)
    budget = torch.randint(0, max_steps + 1, (n,), device="cuda", generator=g)
    act = torch.zeros(n, dtype=torch.int32, device="cuda")
    rew = torch.zeros(n, dtype=torch.float32, device="cuda")
    term = torch.zeros(n, dtype=torch.uint8, device="cuda")
    for t in range(max_steps):
        h.sample_valid_actions(t, act, None)
        act.copy_(torch.where(budget > t, act, torch.full_like(act, -1)))
        h.step(act, rew, term)
    torch.cuda.synchronize()
    return h


def _assert_same(a, b, n_items=None):
    for f in FIELDS:
        x, y = a[f], b[f]
        if n_items is not None:
            x, y = x[:n_items], y[:n_items]
        assert np.array_equal(x, y), f
    m = n_items if n_items is not None else a["mask"].shape[1]
    assert np.array_equal(a["mask"][:, :m], b["mask"][:, :m]), "mask"


@pytest.mark.parametrize("samples", [1, 4])
def test_every_item_equals_host_build(torch, samples):
    n, seed = 4096, 77
    h = _midgame(torch, n, seed)
    st = h.get_state()
    got = _host_view(h.expand(5, samples))
    want = HX.expand(st, seed, 5, samples)
    assert np.array_equal(got["offsets"], want["offsets"])
    _assert_same(got, want)
    # the workload covers deal items, fresh boards and finished games
    deal = ((got["info"] >> 11) & 0x7F) > 0
    counts = np.diff(got["offsets"])
    assert deal.sum() > 1000 and (counts == 0).sum() > 10 and (st["moves"] == 0).sum() > 10
    h.close()


def test_non_deal_items_equal_k1_step_on_replica(torch):
    """Each non-deal item is what bb_env_step (NO_AUTO_RESET) returns on a replica env loaded with the
    same state: ties the expansion to K1 itself."""
    from bbgpu import capi
    n, seed = 512, 13
    h = _midgame(torch, n, seed, rseed=3)
    st = h.get_state()
    ex = _host_view(h.expand(1, 2))
    env_of = np.repeat(np.arange(n), np.diff(ex["offsets"]))
    used = (st["pieces"] >> 24) & 7
    no_deal = np.array([bin(int(u)).count("1") < 2 for u in used], bool)     # more than one piece left
    sel = np.flatnonzero(no_deal[env_of])
    assert (((ex["info"][sel] >> 11) & 0x7F) == 0).all()
    m = sel.size
    assert m > 1000
    r = capi.EnvHandle(m, seed + 1, 0, None, capi.ENV_NO_AUTO_RESET)
    r.set_state(st[env_of[sel]])
    act = torch.as_tensor(ex["action"][sel], device="cuda")
    rew = torch.zeros(m, dtype=torch.float32, device="cuda")
    term = torch.zeros(m, dtype=torch.uint8, device="cuda")
    mask = torch.zeros((3, m), dtype=torch.int64, device="cuda")
    board = torch.zeros(m, dtype=torch.int64, device="cuda")
    pieces = torch.zeros(m, dtype=torch.int32, device="cuda")
    info = torch.zeros(m, dtype=torch.int32, device="cuda")
    r.step(act, rew, term, mask, None, None, info, board, pieces)
    torch.cuda.synchronize()
    assert np.array_equal(rew.cpu().numpy().view(np.uint32), ex["reward"][sel].view(np.uint32))
    assert np.array_equal(term.cpu().numpy(), ex["terminated"][sel])
    assert np.array_equal(info.cpu().numpy().view(np.uint32), ex["info"][sel])
    assert np.array_equal(board.cpu().numpy().view(np.uint64), ex["board"][sel])
    assert np.array_equal(pieces.cpu().numpy().view(np.uint32), ex["pieces"][sel])
    assert np.array_equal(mask.cpu().numpy().view(np.uint64), ex["mask"][:, sel])
    r.close()
    h.close()


def test_no_state_change_and_counter_determinism(torch):
    n, seed = 2048, 5
    h = _midgame(torch, n, seed, rseed=9)
    before = h.get_state()
    a = _host_view(h.expand(7, 3))
    assert h.get_state().tobytes() == before.tobytes()
    b = _host_view(h.expand(7, 3))
    assert np.array_equal(a["offsets"], b["offsets"])
    _assert_same(a, b)
    c = _host_view(h.expand(8, 3))
    assert np.array_equal(a["offsets"], c["offsets"])
    deal = ((a["info"] >> 11) & 0x7F) > 0
    assert deal.any()
    for f in FIELDS:
        assert np.array_equal(a[f][~deal], c[f][~deal]), f
    assert np.array_equal(a["mask"][:, ~deal], c["mask"][:, ~deal])
    assert not np.array_equal(a["pieces"][deal], c["pieces"][deal])
    assert h.get_state().tobytes() == before.tobytes()
    h.close()


def _raw_expand(h, cc, samples, cap, offsets, outs):
    from bbgpu import capi
    p = capi.ptr
    capi.check(capi.lib().bb_env_expand(h.h, cc, samples, cap, p(offsets), *[p(outs.get(f)) for f in FIELDS + ("mask",)],
                                        capi.current_stream()))


@pytest.mark.parametrize("n", [1, 2, 31, 33, 127, 129, 1000, 4097])
def test_expand_stays_inside_its_buffers(torch, n):
    A = Arena(torch)
    h = _midgame(torch, n, 31, max_steps=8, rseed=n)
    dt = {"action": torch.int32, "reward": torch.float32, "terminated": torch.uint8, "info": torch.int32,
          "board": torch.int64, "pieces": torch.int32}
    off0 = A.alloc((n + 1,), torch.int64)
    _raw_expand(h, 2, 4, 0, off0, {})                      # size query
    total = int(off0[n].item())
    assert total > 0
    res = {}
    for cap in (total, max(1, total // 2)):
        off = A.alloc((n + 1,), torch.int64)
        outs = {f: A.alloc((cap,), t) for f, t in dt.items()}
        outs["mask"] = A.alloc((3, cap), torch.int64)
        _raw_expand(h, 2, 4, cap, off, outs)
        A.check()
        assert torch.equal(off, off0)
        res[cap] = {k: v.cpu().numpy() for k, v in outs.items()}
    small = max(1, total // 2)
    for f in FIELDS:
        assert np.array_equal(res[small][f], res[total][f][:small]), f
    assert np.array_equal(res[small]["mask"], res[total]["mask"][:, :small])
    h.close()


def test_large_batch_sampled_envs_equal_host_build(torch):
    n, seed, off = 65536, 1234, 3 * 2 ** 31
    h = _midgame(torch, n, seed, rseed=1, env_offset=off)
    st = h.get_state()
    got = _host_view(h.expand(99, 4))
    rs = np.random.RandomState(0)
    for i in rs.choice(n, 500, replace=False):
        want = HX.expand(st[i:i + 1], seed, 99, 4, env_offset=off + int(i))
        a, b = int(got["offsets"][i]), int(got["offsets"][i + 1])
        assert b - a == want["offsets"][1], i
        for f in FIELDS:
            assert np.array_equal(got[f][a:b], want[f]), (i, f)
        assert np.array_equal(got["mask"][:, a:b], want["mask"]), i
    h.close()


def test_vec_env_expand_modes(torch):
    from bbgpu.vec_env import VectorizedBlockBlastEnv
    for output in ("numpy", "torch"):
        env = VectorizedBlockBlastEnv(64, seed=3, output=output)
        env.reset()
        for _ in range(4):
            env.step(env.sample_valid_actions())
        a, b = env.expand(2), env.expand(2)
        if output == "numpy":
            assert isinstance(a["board"], np.ndarray) and a["board"].dtype == np.uint64 and a["mask"].shape[0] == 3
            assert a["offsets"][-1] == a["action"].shape[0] > 0
        else:
            assert a["board"].is_cuda and int(a["offsets"][-1]) == a["action"].numel() > 0
        env.close()


def _zero_value_agent(torch):
    from bbgpu.ppo import PPOAgent
    torch.manual_seed(1)
    agent = PPOAgent()
    with torch.no_grad():
        for p in agent.network.value_head.parameters():
            p.zero_()
    return agent


def test_lookahead_decision_rule_zero_value_head_equals_brute_force(torch):
    """V = 0: Q is the mean immediate reward; step 0 of evaluate(lookahead=3) must pick, for each env,
    the lowest-index action of maximal f32 reward among the oracle's legal moves."""
    from bbgpu import philox
    from bbgpu.evaluate import evaluate
    from oracle import bb_oracle as O
    agent = _zero_value_agent(torch)
    n, seed = 32, 21
    res = evaluate(agent, num_episodes=n, seed=seed, return_actions=True, lookahead=3, max_steps=1)
    streams = philox.candidate_trios(seed, np.arange(n), 64)
    for i in range(n):
        it = iter(streams[i].tolist())
        env = O.Env(draw=lambda it=it: next(it))
        best, best_a = None, None
        for a in env.valid_actions():
            e2 = copy.deepcopy(env)
            _, r, _, _, _ = e2.step(a)
            q = np.float32(r)
            if best is None or q > best:
                best, best_a = q, a
        assert int(res["actions"][0, i]) == best_a, i


def test_lookahead_chosen_q_matches_independent_recomputation(torch):
    from bbgpu.evaluate import lookahead_actions
    from bbgpu.ppo import PPOAgent
    torch.manual_seed(2)
    agent = PPOAgent()
    agent.eval()
    n, seed = 1024, 8
    h = _midgame(torch, n, seed, rseed=4)
    act, ex, q = lookahead_actions(agent, h, n, 17, 4)
    v = agent.values({"board": ex["board"], "pieces": ex["pieces"], "mask": ex["mask"]}, chunk=65536).reshape(-1).double().cpu().numpy()
    e = _host_view(ex)
    gamma = float(agent.config.gamma)
    act = act.cpu().numpy()
    q = q.cpu().numpy()
    deal_envs = 0
    for i in range(n):
        a0, a1 = int(e["offsets"][i]), int(e["offsets"][i + 1])
        if a0 == a1:
            continue
        qi = e["reward"][a0:a1].astype(np.float64) + gamma * (1.0 - e["terminated"][a0:a1]) * v[a0:a1]
        acts = e["action"][a0:a1]
        per = {int(a): qi[acts == a].mean() for a in np.unique(acts)}
        deal_envs += (acts.size > len(per))
        best = max(per.values())
        assert abs(per[int(act[i])] - best) < 1e-5 * max(1.0, abs(best)), i
        assert abs(q[i, act[i]] - per[int(act[i])]) < 1e-5 * max(1.0, abs(best)), i
        assert np.isneginf(q[i][[a for a in range(192) if a not in per]]).all()
    assert deal_envs > 50
    h.close()


def test_lookahead_evaluation_replays_through_the_oracle(torch):
    """evaluate(lookahead=2): the logged actions replay through the Python oracle fed the same trio
    streams — final score, length, lines, max combo and summed reward identical, no rejected action."""
    from bbgpu import philox
    from bbgpu.evaluate import evaluate
    from bbgpu.ppo import PPOAgent
    from oracle import bb_oracle as O
    torch.manual_seed(5)
    agent = PPOAgent()
    n, seed = 48, 9
    res = evaluate(agent, num_episodes=n, seed=seed, return_actions=True, lookahead=2)
    assert res["finished"] == n and res["actions"].shape[1] == n
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
        assert info["score"] == res["scores"][i] and info["moves"] == res["lengths"][i] == t, (i, info, res["scores"][i])
        assert info["lines_cleared"] == res["lines"][i] and info["max_combo"] == res["max_combos"][i]
        assert abs(total - res["rewards_per_episode"][i]) < 1e-4 * max(1.0, abs(total))
