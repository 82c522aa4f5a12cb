"""CPU checks of the board symmetries (group D4) the symmetric policy rests on: the generated tables against a
fresh derivation from oracle/piece_table.json, the group laws of bb_sym_* (host build of bb_rules.cuh), the
anchor map against the oracle's placement rule, the equivariance of one env step (host build and oracle) under
every symmetry with the candidate stream mapped through the piece permutation, and the eight views of the
observation against the oracle's obs() of the transformed game."""
import os
import sys

import numpy as np
import pytest

import hostsym as S
from bbgpu import philox
from oracle import bb_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = 97531

# the symmetry ids of bb_rules.cuh as maps of cell (r, c)
CELL = (lambda r, c: (r, c), lambda r, c: (c, 7 - r), lambda r, c: (7 - r, 7 - c), lambda r, c: (7 - c, r),
        lambda r, c: (r, 7 - c), lambda r, c: (7 - r, c), lambda r, c: (c, r), lambda r, c: (7 - c, 7 - r))


def _grid_sym(g, grid):
    out = O.new_grid()
    for r in range(8):
        for c in range(8):
            rr, cc = CELL[g](r, c)
            out[rr][cc] = grid[r][c]
    return out


def _board_sym_loop(g, b):
    out = 0
    for a in range(64):
        if (b >> a) & 1:
            r, c = CELL[g](a >> 3, a & 7)
            out |= 1 << (r * 8 + c)
    return out


def _fresh_tables():
    """perm / shift derived here from the piece cells: image of the piece drawn on a grid, normalised."""
    shapes = {frozenset(cells): p for p, cells in enumerate(O.PIECE_CELLS)}
    perm, shift = np.zeros((8, 37), np.int64), np.zeros((8, 37), np.int64)
    for g in range(8):
        for p, cells in enumerate(O.PIECE_CELLS):
            img = [CELL[g](r, c) for r, c in cells]
            r0, c0 = min(r for r, _ in img), min(c for _, c in img)
            perm[g, p] = shapes[frozenset((r - r0, c - c0) for r, c in img)]
            # anchor (0, 0): its image cell minus the top-left of the image of the bounding box
            box = [CELL[g](r, c) for r in range(O.PIECE_H[p]) for c in range(O.PIECE_W[p])]
            ar, ac = CELL[g](0, 0)
            shift[g, p] = 8 * (ar - min(r for r, _ in box)) + (ac - min(c for _, c in box))
    return perm, shift


def _compose(g, h):
    """k with CELL[k] = CELL[g] after CELL[h]"""
    for k in range(8):
        if all(CELL[k](r, c) == CELL[g](*CELL[h](r, c)) for r in range(8) for c in range(8)):
            return k
    raise AssertionError((g, h))


def test_tables_match_a_fresh_derivation_and_are_permutations(tmp_path):
    perm, shift = S.tables()
    fp, fs = _fresh_tables()
    assert np.array_equal(perm[:, :37], fp) and np.array_equal(shift[:, :37], fs)
    assert np.array_equal(perm[:, 37:], np.tile(np.arange(37, 40), (8, 1))) and not shift[:, 37:].any()
    for g in range(8):
        assert sorted(perm[g, :37].tolist()) == list(range(37)), g
        # the image keeps the cell count; h and w swap exactly when the map transposes
        for p in range(37):
            q = perm[g, p]
            assert len(O.PIECE_CELLS[q]) == len(O.PIECE_CELLS[p])
            hw = (O.PIECE_H[p], O.PIECE_W[p])
            assert (O.PIECE_H[q], O.PIECE_W[q]) == (hw[::-1] if g in (1, 3, 6, 7) else hw)
    # the committed include is what the generator writes now
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import gen_piece_tables as G
    finally:
        sys.path.pop(0)
    rows = [dict(index=i, cells=[list(c) for c in cells], h=O.PIECE_H[i], w=O.PIECE_W[i])
            for i, cells in enumerate(O.PIECE_CELLS)]
    out = tmp_path / "bb_sym_table.inc"
    G.write_sym_inc(rows, str(out))
    committed = os.path.join(ROOT, "block-blast-ai---reinforcement-learning-agent_b200", "csrc", "bb_sym_table.inc")
    assert out.read_bytes() == open(committed, "rb").read()


def test_group_laws_of_the_host_build():
    rs = np.random.RandomState(1)
    boards = [int(x) for x in rs.randint(0, 2 ** 63, 200, dtype=np.int64).astype(np.uint64)] + [0, 2 ** 64 - 1, 1, 1 << 63]
    boards += [int(b) | (1 << 63) for b in boards[:50]]
    # bb_sym_cell and bb_sym_board equal the cell maps
    for g in range(8):
        for a in range(64):
            r, c = CELL[g](a >> 3, a & 7)
            assert S.sym_cell(g, a) == r * 8 + c
        for b in boards:
            assert S.sym_board(g, b) == _board_sym_loop(g, b), (g, hex(b))
    assert all(S.sym_board(0, b) == b for b in boards)
    assert all(S.sym_pieces(0, pw) == pw for pw in rs.randint(0, 2 ** 31, 100).tolist())
    # composition table from the host cell maps == composition of the spec's cell maps; it is a group table
    table = np.zeros((8, 8), np.int64)
    for g in range(8):
        for h in range(8):
            host = [S.sym_cell(g, S.sym_cell(h, a)) for a in range(64)]
            k = [k for k in range(8) if [S.sym_cell(k, a) for a in range(64)] == host]
            assert k == [_compose(g, h)], (g, h)
            table[g, h] = k[0]
            for b in boards[:40]:
                assert S.sym_board(g, S.sym_board(h, b)) == S.sym_board(k[0], b)
            pw = int(rs.randint(0, 37 ** 3)) % 37 | (int(rs.randint(37)) << 8) | (int(rs.randint(37)) << 16) | (5 << 24)
            assert S.sym_pieces(g, S.sym_pieces(h, pw)) == S.sym_pieces(k[0], pw)
    for g in range(8):
        assert sorted(table[g].tolist()) == list(range(8)) and sorted(table[:, g].tolist()) == list(range(8))
        inv = [h for h in range(8) if table[g, h] == 0]
        assert len(inv) == 1 and table[inv[0], g] == 0
        for b in boards[:40]:
            assert S.sym_board(inv[0], S.sym_board(g, b)) == b
    # ids >= 37 in a used slot and the used bits stay as they are
    assert S.sym_pieces(1, 0x07FF2500 | 0x1) == (0x07FF2500 & 0xFFFF0000) | (S.sym_pieces(1, 0x2501) & 0xFFFF)


def test_legal_anchors_map_to_legal_anchors_of_the_image_piece():
    rs = np.random.RandomState(2)
    grids = [O.new_grid()]
    for density in (0.15, 0.3, 0.45):
        for _ in range(2):
            grids.append([[int(rs.rand() < density) for _ in range(8)] for _ in range(8)])
    perm, _ = S.tables()
    for grid in grids:
        for g in range(8):
            tg = _grid_sym(g, grid)
            for p in range(37):
                q = int(perm[g, p])
                legal = [r * 8 + c for r in range(8) for c in range(8) if O.fits(grid, p, r, c)]
                legal_img = {r * 8 + c for r in range(8) for c in range(8) if O.fits(tg, q, r, c)}
                img = [S.sym_anchor(g, p, a) for a in legal]
                assert len(set(img)) == len(img) and set(img) == legal_img, (g, p)
                plane = sum(1 << a for a in legal)
                assert S.sym_mask_plane(g, p, plane) == sum(1 << a for a in legal_img), (g, p)


def _draw(trios):
    it = iter(np.asarray(trios).tolist())
    return lambda: next(it)


def _set_oracle(env, board, trio, used, src, rec):
    """oracle env in the state of a host record (board / trio / used given), drawing from ``src``"""
    g = env.game
    g.grid = O.u64_to_grid(int(board))
    g.trio, g.used = [int(x) for x in trio], [bool(u) for u in used]
    g.score, g.streak, g.moves = int(rec["score"]), int(rec["streak"]), int(rec["moves"])
    g.lines_total, g.max_streak, g.blocks_total = int(rec["lines_total"]), int(rec["max_streak"]), int(rec["blocks_total"])
    g.over = bool((int(rec["aux"]) >> 16) & 1)
    g.draw = _draw(src)
    env.prev_holes = int(rec["aux"]) & 0xFF
    env.prev_center = 1.0 - ((int(rec["aux"]) >> 8) & 0xFF) / 16.0


def _legal(state):
    """legal actions of a host record (the mask of an invalid step is the unchanged state's)"""
    _, _, _, info, m = S.step(state, -1, np.zeros((1, 3), np.uint8))
    assert info == 1
    return [k * 64 + a for k in range(3) for a in range(64) if (int(m[k]) >> a) & 1]


@pytest.fixture(scope="module")
def played_states():
    """~60 host records after 0..40 random legal moves (streams drawn from Philox), with a fresh candidate
    stream each for the step under test"""
    import hostrules as H
    rs = np.random.RandomState(3)
    n = 60
    streams = philox.candidate_trios(SEED, np.arange(n), 400)
    out = []
    for i in range(n):
        t = streams[i]
        s = np.zeros((), H.STATE_DTYPE)
        s["pieces"] = int(t[0, 0]) | (int(t[0, 1]) << 8) | (int(t[0, 2]) << 16)
        s["draw_ctr"] = 1
        for _ in range(int(rs.randint(0, 41))):
            legal = _legal(s)
            if not legal:
                break
            s, _, term, _, _ = S.step(s, legal[rs.randint(len(legal))], t)
            if term:
                break
        out.append(s)
    return out


def test_one_step_is_equivariant_under_every_symmetry(played_states):
    """For every state, symmetry g and legal action: stepping the transformed state with the mapped action on
    the candidate stream mapped through PERM gives the transformed successor, mapped trio and mask, the same
    info word and the same reward bits — in the host build of the rules and in the oracle."""
    rs = np.random.RandomState(4)
    perm, _ = S.tables()
    checked = 0
    for s in played_states:
        legal = _legal(s)
        if not legal:
            continue
        s = s.copy()
        s["draw_ctr"] = 0                           # the step under test deals from the start of `src`
        for a in [legal[k] for k in rs.choice(len(legal), min(3, len(legal)), replace=False)]:
            src = rs.randint(0, 37, (100, 3)).astype(np.uint8)
            s1, r1, t1, i1, m1 = S.step(s, a, src)
            pw, pw1 = int(s["pieces"]), int(s1["pieces"])
            # the host step is the oracle's step
            env = O.Env(draw=_draw(src))
            _set_oracle(env, s["board"], [(pw >> 8 * k) & 0xFF for k in range(3)],
                        [(pw >> 24 + k) & 1 for k in range(3)], src, s)
            obs, rew, term, _, _ = env.step(a)
            assert O.grid_to_u64(env.game.grid) == int(s1["board"]) and env.game.trio == [(pw1 >> 8 * k) & 0xFF for k in range(3)]
            assert np.float32(rew).view(np.uint32) == np.float32(r1).view(np.uint32) and int(term) == t1
            for g in range(1, 8):
                sg = s.copy()
                sg["board"] = S.sym_board(g, int(s["board"]))
                sg["pieces"] = S.sym_pieces(g, pw)
                srcg = perm[g][src]
                ag = S.sym_action(g, pw, a)
                s1g, r1g, t1g, i1g, m1g = S.step(sg, ag, srcg)
                assert int(s1g["board"]) == S.sym_board(g, int(s1["board"])), (g, a)
                assert int(s1g["pieces"]) == S.sym_pieces(g, pw1), (g, a)
                for k in range(3):
                    assert int(m1g[k]) == S.sym_mask_plane(g, (pw1 >> 8 * k) & 0xFF, int(m1[k])), (g, a, k)
                assert i1g == i1 and t1g == t1
                assert np.float32(r1g).view(np.uint32) == np.float32(r1).view(np.uint32)
                for f in ("score", "streak", "moves", "lines_total", "max_streak", "blocks_total", "aux", "draw_ctr"):
                    assert s1g[f] == s1[f], f
                # the oracle on the transformed game: same float64 reward, transformed board
                eg = O.Env(draw=_draw(srcg))
                pwg = int(sg["pieces"])
                _set_oracle(eg, sg["board"], [(pwg >> 8 * k) & 0xFF for k in range(3)],
                            [(pwg >> 24 + k) & 1 for k in range(3)], srcg, s)
                _, rewg, termg, _, _ = eg.step(ag)
                assert np.float64(rewg).view(np.uint64) == np.float64(rew).view(np.uint64) and termg == term
                assert O.grid_to_u64(eg.game.grid) == int(s1g["board"])
                checked += 1
    assert checked > 500


def test_eight_views_equal_the_oracle_obs_of_the_transformed_game(played_states):
    perm, _ = S.tables()
    board = np.array([int(s["board"]) for s in played_states], np.uint64)
    pieces = np.array([int(s["pieces"]) for s in played_states], np.uint32)
    # one row with an out-of-range id in a used slot and one in an unused slot (both give an empty plane)
    board = np.append(board, [np.uint64(0x8000000000000001)] * 2)
    pieces = np.append(pieces, [np.uint32(0x01280203), np.uint32(0x00280203)])
    views = S.obs_views(board, pieces)
    for i in range(len(played_states)):
        pw = int(pieces[i])
        for g in range(8):
            env = O.Env(draw=_draw(np.zeros((1, 3), np.uint8)))
            env.game.grid = _grid_sym(g, O.u64_to_grid(int(board[i])))
            env.game.trio = [int(perm[g, (pw >> 8 * k) & 0xFF]) for k in range(3)]
            env.game.used = [bool((pw >> 24 + k) & 1) for k in range(3)]
            o = env.obs()
            bits = lambda plane: sum(1 << a for a in range(64) if plane.reshape(-1)[a])
            assert int(views[g, i, 0]) == bits(o["board"]), (i, g)
            for k in range(3):
                assert int(views[g, i, 1 + k]) == bits(o["pieces"][k]), (i, g, k)
    i = len(played_states)
    for g in range(8):
        assert int(views[g, i, 0]) == int(views[g, i + 1, 0]) == S.sym_board(g, 0x8000000000000001)
        # 0x01280203: slot 0 used, slot 2 holds id 40; 0x00280203: only slot 2 holds id 40
        assert views[g, i, 1] == 0 and views[g, i, 3] == 0 and views[g, i + 1, 3] == 0
        assert views[g, i, 2] == views[g, i + 1, 2] == sum(1 << (r * 8 + c) for r, c in O.PIECE_CELLS[int(perm[g, 2])])
        assert views[g, i + 1, 1] != 0


def test_c_abi_rejects_bad_arguments_of_the_symmetry_entry_points():
    """argument checks of bb_unpack_obs_sym / bb_sym_logits_mean[_backward] (they run before any launch)"""
    import ctypes as C
    from bbgpu import capi
    L = capi.lib()
    err = lambda: L.bb_last_error().decode()
    assert L.bb_unpack_obs_sym(None, None, None, None, 0, -1, None) == -1 and "negative n" in err()
    assert L.bb_unpack_obs_sym(None, None, None, None, 7, 4, None) == -1 and "obs_dtype" in err()
    assert L.bb_unpack_obs_sym(None, None, None, None, 0, 4, None) == -1 and "required" in err()
    assert L.bb_unpack_obs_sym(None, None, None, None, 0, 0, None) == 0
    assert L.bb_sym_logits_mean(None, 2, None, None, 4, None) == -1 and "logits_dtype" in err()
    assert L.bb_sym_logits_mean(None, 0, None, None, 4, None) == -1 and "NULL" in err()
    # 16-byte vector accesses: a misaligned logits / grad_logits pointer is refused, not dereferenced
    assert L.bb_sym_logits_mean(C.c_void_p(0x1008), 0, C.c_void_p(0x2000), C.c_void_p(0x3000), 4, None) == -1
    assert "aligned" in err()
    assert L.bb_sym_logits_mean_backward(C.c_void_p(0x2000), C.c_void_p(0x2000), C.c_void_p(0x1004), 1, 4, None) == -1
    assert "aligned" in err()
    assert L.bb_sym_logits_mean_backward(None, None, None, 0, 0, None) == 0
