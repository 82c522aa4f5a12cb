"""ctypes loader for the host build of the canonical view (tests/hostbuild/bb_canon_host.cpp: bb_sym_canonical of
the product's rules header compiled for the host).  Test infrastructure only.  The library is compiled into a
private temporary directory on first use, so the tests work from a read-only tree."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_TESTS = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_TESTS, "hostbuild", "bb_canon_host.cpp")
_CSRC = os.path.join(os.path.dirname(_TESTS), "block-blast-ai---reinforcement-learning-agent_b200", "csrc")
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        out = tempfile.mkdtemp(prefix="bbc_")
        atexit.register(shutil.rmtree, out, True)
        so = os.path.join(out, "libbbcanon_host.so")
        gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.check_call([gxx, "-O2", "-fPIC", "-ffp-contract=off", "-std=c++17", "-I" + _CSRC, "-x", "c++",
                               "-shared", "-o", so, _SRC], stderr=subprocess.DEVNULL)
        L = C.CDLL(so)
        L.bbc_canonical.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
        _LIB = L
    return _LIB


def canonical(board, pieces):
    """(board uint64 [n], pieces uint32 [n], views uint8 [n]): canonical view and view set of packed rows."""
    b = np.ascontiguousarray(board, np.uint64)
    p = np.ascontiguousarray(pieces, np.uint32)
    n = b.shape[0]
    bo, po, v = np.zeros(n, np.uint64), np.zeros(n, np.uint32), np.zeros(n, np.uint8)
    p_ = lambda a: a.ctypes.data_as(C.c_void_p)
    lib().bbc_canonical(p_(b), p_(p), C.c_int64(n), p_(bo), p_(po), p_(v))
    return bo, po, v


def restated(board, pieces):
    """numpy restatement of the definition over hostsym.sym_rows: the view with the smallest (board u64, pieces
    u32) key, and the mask of the views equal to it."""
    import hostsym as S
    n = len(board)
    vb = np.stack([S.sym_rows(g, board, pieces)[0] for g in range(8)])            # [8, n]
    vp = np.stack([S.sym_rows(g, board, pieces)[1] for g in range(8)])
    best = np.zeros(n, np.int64)
    for g in range(1, 8):
        cb, cp = vb[best, np.arange(n)], vp[best, np.arange(n)]
        less = (vb[g] < cb) | ((vb[g] == cb) & (vp[g] < cp))
        best = np.where(less, g, best)
    cb, cp = vb[best, np.arange(n)], vp[best, np.arange(n)]
    views = np.zeros(n, np.uint8)
    for g in range(8):
        views |= (((vb[g] == cb) & (vp[g] == cp)).astype(np.uint8) << np.uint8(g))
    return cb, cp, views


def random_rows(n, rs):
    """random packed rows: any board, ids 0..36 (and a few >= 37), random used bits"""
    board = rs.randint(0, 2 ** 63, n, dtype=np.int64).astype(np.uint64) | (rs.randint(0, 2, n).astype(np.uint64) << np.uint64(63))
    ids = rs.randint(0, 37, (n, 3))
    ids[rs.rand(n, 3) < 0.02] = 40 + rs.randint(0, 200)
    used = (rs.rand(n, 3) < 0.3).astype(np.int64)
    return board, pack(ids, used)


def pack(ids, used):
    ids, used = np.asarray(ids, np.int64), np.asarray(used, np.int64)
    return (ids[:, 0] | (ids[:, 1] << 8) | (ids[:, 2] << 16) | (used[:, 0] << 24) | (used[:, 1] << 25)
            | (used[:, 2] << 26)).astype(np.uint32)


#: subgroups of D4 (ids of bb_rules.cuh) used to build states with a known stabiliser
SUBGROUPS = [(0,), (0, 6), (0, 7), (0, 2), (0, 4), (0, 5), (0, 1, 2, 3), (0, 2, 4, 5), (0, 2, 6, 7), tuple(range(8))]


def symmetric_rows(n, subgroup, rs):
    """n packed rows each fixed by every symmetry of ``subgroup``: the board is the union of the subgroup's images
    of a few random cells (or empty), the pieces are ids that every element of the subgroup fixes (BB_SYM_PERM);
    used bits random."""
    import hostsym as S
    perm, _ = S.tables()
    fixed = [p for p in range(37) if all(perm[g][p] == p for g in subgroup)]
    board = np.zeros(n, np.uint64)
    for i in range(n):
        if rs.rand() < 0.2:
            continue
        b0 = 0
        for c in rs.randint(0, 64, rs.randint(1, 6)):
            b0 |= 1 << int(c)
        b = 0
        for g in subgroup:
            b |= S.sym_board(g, b0)
        board[i] = b
    ids = np.asarray(fixed)[rs.randint(0, len(fixed), (n, 3))]
    return board, pack(ids, rs.rand(n, 3) < 0.3)
