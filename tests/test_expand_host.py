"""CPU-only checks of the one-ply expansion (bb_env_expand): the host build of its per-item body
(bbx_expand: the same bb_rules.cuh code, with the sequential deal on the LOOKAHEAD stream) against
the Python oracle stepping a copy of each env with every legal action, the LOOKAHEAD stream against
its numpy replica, and the C ABI's argument checks (no GPU needed)."""
import copy
import ctypes as C

import numpy as np
import pytest

import hostexpand as HX
import hostrules as H
from bbgpu import philox
from oracle import bb_oracle as O

SEED = 20240611


def _stream_draw(trios):
    """oracle ``draw`` callable over a fixed [L, 3] candidate array."""
    it = iter(trios.tolist())
    return lambda: next(it)


def _info_word(res, draws):
    return (res["lines"] << 1) | (res["blocks"] << 4) | (res["combo_mult"] << 8) | (draws << 11) | (res["gain"] << 18)


@pytest.fixture(scope="module")
def midgame():
    """~300 envs driven by seeded random play to 0..70 moves (some finish: NO_AUTO_RESET keeps them
    GAME_OVER); the host build and the Python oracle play the same moves."""
    n = 300
    rs = np.random.RandomState(7)
    streams = philox.candidate_trios(SEED, np.arange(n), 400)
    envs = [O.Env(draw=_stream_draw(streams[i])) for i in range(n)]
    host = H.HostEnv(n, SEED, flags=2)          # BB_ENV_NO_AUTO_RESET
    target = rs.randint(0, 71, n)
    target[:10] = 0                             # fresh boards (0 filled cells)
    for t in range(int(target.max())):
        m = host.masks()
        acts = np.full(n, -1, np.int32)         # invalid = no-op in both implementations
        for i in range(n):
            va = [p * 64 + k for p in range(3) for k in range(64) if (int(m[i, p]) >> k) & 1]
            if t < target[i] and va:
                acts[i] = va[rs.randint(len(va))]
        host.step(acts)
        for i in range(n):
            if acts[i] >= 0:
                envs[i].step(int(acts[i]))
    for i in range(n):
        assert O.grid_to_u64(envs[i].game.grid) == int(host.state["board"][i])
    return host, envs


def test_expansion_equals_oracle_step_of_every_legal_move(midgame):
    host, envs = midgame
    n, K, cc = len(envs), 3, 11
    ex = HX.expand(host.state, SEED, cc, K)
    off = ex["offsets"]
    fills, n_deal, n_over = [], 0, 0
    for i, env in enumerate(envs):
        g = env.game
        fills.append(g.filled())
        mask = g.mask3().reshape(-1)
        acts = np.flatnonzero(mask) if not g.over else np.zeros(0, np.int64)
        deal = sum(g.used) == 2
        per = K if deal else 1
        assert off[i + 1] - off[i] == len(acts) * per, i
        n_over += g.over
        j = int(off[i])
        for a in acts:
            for k in range(per):
                e2 = copy.deepcopy(env)
                if deal:
                    e2.game.draw = _stream_draw(philox.lookahead_trios(SEED, [i], cc, k, 100)[0])
                d0 = e2.game.draws
                res = e2.game.move(*O.Env.decode(int(a)))
                r = np.float32(e2.reward(res))
                g2 = e2.game
                assert ex["action"][j] == a
                assert ex["board"][j] == O.grid_to_u64(g2.grid), (i, a, k)
                pw = g2.trio[0] | (g2.trio[1] << 8) | (g2.trio[2] << 16) | (sum(u << p for p, u in enumerate(g2.used)) << 24)
                assert ex["pieces"][j] == pw, (i, a, k)
                m2 = g2.mask3().reshape(3, 64)
                for p in range(3):
                    assert int(ex["mask"][p, j]) == sum(1 << int(b) for b in np.flatnonzero(m2[p])), (i, a, k, p)
                assert ex["reward"][j].view(np.uint32) == r.view(np.uint32), (i, a, k)
                assert ex["terminated"][j] == int(res["game_over"]), (i, a, k)
                assert ex["info"][j] == _info_word(res, g2.draws - d0), (i, a, k)
                n_deal += deal
                j += 1
        assert j == off[i + 1]
    assert off[n] == len(ex["action"])
    # coverage: fresh and half-full boards, one-piece-left states (deal items) and finished games
    assert min(fills) == 0 and max(fills) >= 40, (min(fills), max(fills))
    assert n_deal >= 300 and n_over >= 5, (n_deal, n_over)


def test_expansion_does_not_depend_on_capacity_and_counter_moves_only_deal_items(midgame):
    host, _ = midgame
    full = HX.expand(host.state, SEED, 3, 2)
    total = int(full["offsets"][-1])
    part = HX.expand(host.state, SEED, 3, 2, capacity=total // 3)
    assert np.array_equal(part["offsets"], full["offsets"])
    for f in HX.EXPAND_FIELDS:
        assert np.array_equal(part[f], full[f][:total // 3]), f
    other = HX.expand(host.state, SEED, 4, 2)
    deal = (full["info"] >> 11) & 0x7F > 0
    assert deal.any() and np.array_equal(other["offsets"], full["offsets"])
    for f in HX.EXPAND_FIELDS:
        assert np.array_equal(other[f][~deal], full[f][~deal]), f
    assert not np.array_equal(other["pieces"][deal], full["pieces"][deal])


def test_lookahead_stream_equals_numpy_replica():
    for seed in (0, SEED, 2 ** 63 + 12345):
        for env in (0, 5, 2 ** 33 + 7):
            for cc in (0, 1, 2 ** 25 - 1):
                for k in (0, 1, 63):
                    want = philox.lookahead_trios(seed, [env], cc, k, 100)[0]
                    for d in (0, 1, 50, 99):
                        w = HX.lookahead_trio(seed, env, cc, k, d)
                        assert [w & 0xFF, (w >> 8) & 0xFF, (w >> 16) & 0xFF] == want[d].tolist()
    # distinct from the env's own TRIO stream at the same counter words
    a = philox.lookahead_trios(1, np.arange(64), 0, 0, 8)
    assert not np.array_equal(a, philox.candidate_trios(1, np.arange(64), 8))


def test_expand_abi_error_paths_return_codes_not_crashes():
    """Argument errors come back before any CUDA call (this runs without a GPU).  A zeroed host
    buffer stands in for the env: the argument checks reject the call before the env is read."""
    import bbgpu.build as b
    lib = C.CDLL(b.build())
    lib.bb_last_error.restype = C.c_char_p
    vp, i64, u64, i32 = C.c_void_p, C.c_int64, C.c_uint64, C.c_int32
    lib.bb_env_expand.argtypes = [vp, u64, i32, i64] + [vp] * 9
    fake = (C.c_char * 512)()
    off = (C.c_int64 * 4)()
    rest = [None] * 8
    assert lib.bb_env_expand(None, 0, 1, 0, off, *rest) < 0 and b"env is NULL" in lib.bb_last_error()
    assert lib.bb_env_expand(fake, 0, 1, 0, None, *rest) < 0 and b"offsets" in lib.bb_last_error()
    for s in (0, -1, 65):
        assert lib.bb_env_expand(fake, 0, s, 0, off, *rest) < 0 and b"samples" in lib.bb_last_error()
    assert lib.bb_env_expand(fake, 2 ** 25, 1, 0, off, *rest) < 0 and b"call_counter" in lib.bb_last_error()
    assert lib.bb_env_expand(fake, 2 ** 64 - 1, 1, 0, off, *rest) < 0 and b"call_counter" in lib.bb_last_error()
    assert lib.bb_env_expand(fake, 0, 1, -1, off, *rest) < 0 and b"capacity" in lib.bb_last_error()
