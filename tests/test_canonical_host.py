"""CPU checks of the canonical view (bb_sym_canonical, csrc/bb_rules.cuh, host build): against a numpy restatement
of its definition on random states and on states with stabilisers of order 2, 4 and 8, its invariance under the
eight symmetries and the transformation law of its view set, and the C ABI's argument checks of the canonical-frame
entry points."""
import ctypes as C

import numpy as np
import pytest

import hostcanon as K
import hostsym as S


def _compose():
    """comp[a][b] = the symmetry id of T_a o T_b (apply b, then a), read off bb_sym_board on a board that no
    symmetry fixes"""
    b = 0x107                         # cells (0,0) (0,1) (0,2) (1,0): no symmetry maps it onto itself
    imgs = [S.sym_board(g, b) for g in range(8)]
    assert len(set(imgs)) == 8
    return np.array([[imgs.index(S.sym_board(a, S.sym_board(g, b))) for g in range(8)] for a in range(8)])


def _check(board, pieces):
    cb, cp, v = K.canonical(board, pieces)
    rb, rp, rv = K.restated(board, pieces)
    assert np.array_equal(cb, rb) and np.array_equal(cp, rp) and np.array_equal(v, rv)
    return cb, cp, v


def test_canonical_view_matches_restatement_on_random_states():
    rs = np.random.RandomState(0)
    board, pieces = K.random_rows(20000, rs)
    _check(board, pieces)
    # sparse boards and empty boards: ties on the board word, decided by the pieces word
    sparse = np.array([sum(1 << int(c) for c in rs.randint(0, 64, rs.randint(0, 3))) for _ in range(5000)], np.uint64)
    _, v = _check(sparse, pieces[:5000])[1:]
    assert (v != 1).any()


@pytest.mark.parametrize("subgroup", K.SUBGROUPS)
def test_view_set_is_the_stabiliser_on_constructed_states(subgroup):
    rs = np.random.RandomState(len(subgroup) * 10 + subgroup[-1])
    board, pieces = K.symmetric_rows(2000, subgroup, rs)
    _, _, v = _check(board, pieces)
    size = np.array([bin(int(x)).count("1") for x in v])
    assert (size % len(subgroup) == 0).all()                   # the stabiliser contains the subgroup
    assert (size == len(subgroup)).mean() > 0.5                # and mostly is it
    if len(subgroup) == 8:
        assert (v == 0xFF).all()


def test_empty_board_with_a_fully_symmetric_trio_has_eight_views():
    perm, _ = S.tables()
    assert all(perm[g][p] == p for g in range(8) for p in (0, 17, 36))
    _, _, v = _check(np.zeros(1, np.uint64), K.pack([[0, 17, 36]], [[0, 0, 0]]))
    assert v[0] == 0xFF


def test_canonical_view_is_invariant_and_view_set_transforms():
    """c(k.s) = c(s) and M(k.s) = M(s).k^-1 (bit g of M(k.s) set iff g o k is in M(s)) for every k; |M| * |orbit| = 8"""
    comp = _compose()
    rs = np.random.RandomState(3)
    parts = [K.random_rows(3000, rs)] + [K.symmetric_rows(500, h, rs) for h in K.SUBGROUPS[1:]]
    board = np.concatenate([b for b, _ in parts])
    pieces = np.concatenate([p for _, p in parts])
    cb, cp, v = K.canonical(board, pieces)
    for k in range(8):
        bk, pk = S.sym_rows(k, board, pieces)
        cbk, cpk, vk = K.canonical(bk, pk)
        assert np.array_equal(cbk, cb) and np.array_equal(cpk, cp), k
        want = np.zeros_like(v)
        for g in range(8):
            want |= (((v >> np.uint8(comp[g][k])) & np.uint8(1)) << np.uint8(g)).astype(np.uint8)
        assert np.array_equal(vk, want), k
    views = np.stack([np.stack(S.sym_rows(g, board, pieces)).astype(np.uint64) for g in range(8)])   # [8, 2, n]
    orbit = np.array([len({(int(views[g, 0, i]), int(views[g, 1, i])) for g in range(8)}) for i in range(len(board))])
    size = np.array([bin(int(x)).count("1") for x in v])
    assert (size * orbit == 8).all()
    assert set(size) == {1, 2, 4, 8}


@pytest.fixture(scope="module")
def libpath():
    import bbgpu.build as b
    return b.build()


def test_c_abi_rejects_bad_arguments_of_the_canonical_entry_points(libpath):
    from bbgpu import capi
    lib = capi.lib()
    one = C.c_void_p(16)                                        # never dereferenced: every call fails its checks
    odd = C.c_void_p(24)                                        # not 16-byte aligned
    assert lib.bb_sym_canonical(one, one, None, one, one, one, -1, None) == -1 and b"negative" in lib.bb_last_error()
    assert lib.bb_sym_canonical(one, None, None, one, one, one, 4, None) == -1 and b"NULL" in lib.bb_last_error()
    assert lib.bb_sym_canonical(one, one, None, one, one, None, 4, None) == -1 and b"NULL" in lib.bb_last_error()
    assert lib.bb_sym_canonical(None, None, None, None, None, None, 0, None) == 0
    f = lib.bb_sym_logits_canonical
    assert f(one, 0, one, one, one, -1, None) == -1 and b"negative" in lib.bb_last_error()
    assert f(one, 5, one, one, one, 4, None) == -1 and b"dtype" in lib.bb_last_error()
    assert f(one, 0, one, None, one, 4, None) == -1 and b"NULL" in lib.bb_last_error()
    assert f(odd, 1, one, one, one, 4, None) == -1 and b"aligned" in lib.bb_last_error()
    b = lib.bb_sym_logits_canonical_backward
    assert b(one, one, one, one, 0, -1, None) == -1 and b"negative" in lib.bb_last_error()
    assert b(one, one, one, one, 2, 4, None) == -1 and b"dtype" in lib.bb_last_error()
    assert b(one, None, one, one, 0, 4, None) == -1 and b"NULL" in lib.bb_last_error()
    assert b(one, one, one, odd, 1, 4, None) == -1 and b"aligned" in lib.bb_last_error()
    assert b(odd, one, one, one, 0, 4, None) == -1 and b"aligned" in lib.bb_last_error()
