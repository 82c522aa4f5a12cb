"""ctypes loader for the host build of the board symmetries (tests/hostbuild/bb_sym_host.cpp: bb_sym_* of the
product's rules header compiled for the host, plus one env step on an injected candidate stream).  Test
infrastructure only.  The library is compiled into a private temporary directory on first use, so the tests
work from a read-only tree."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from hostrules import STATE_DTYPE

_TESTS = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_TESTS, "hostbuild", "bb_sym_host.cpp")
_CSRC = os.path.join(os.path.dirname(_TESTS), "block-blast-ai---reinforcement-learning-agent_b200", "csrc")
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        out = tempfile.mkdtemp(prefix="bbs_")
        atexit.register(shutil.rmtree, out, True)
        so = os.path.join(out, "libbbsym_host.so")
        gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        # the flags of tests/hostbuild/Makefile (no FMA contraction: the float64 reward must be bit-exact)
        subprocess.check_call([gxx, "-O2", "-fPIC", "-ffp-contract=off", "-std=c++17", "-I" + _CSRC, "-x", "c++",
                               "-shared", "-o", so, _SRC], stderr=subprocess.DEVNULL)
        L = C.CDLL(so)
        L.bbs_state_size.restype = C.c_int64
        L.bbs_sym_board.restype = C.c_uint64
        L.bbs_sym_board.argtypes = [C.c_int, C.c_uint64]
        L.bbs_sym_cell.argtypes = [C.c_int, C.c_int]
        L.bbs_sym_pieces.restype = C.c_uint32
        L.bbs_sym_pieces.argtypes = [C.c_int, C.c_uint32]
        L.bbs_sym_anchor.argtypes = [C.c_int, C.c_uint32, C.c_int]
        L.bbs_sym_mask_plane.restype = C.c_uint64
        L.bbs_sym_mask_plane.argtypes = [C.c_int, C.c_uint32, C.c_uint64]
        L.bbs_step.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                               C.c_void_p, C.c_void_p]
        assert L.bbs_state_size() == STATE_DTYPE.itemsize == 48
        _LIB = L
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def tables():
    """(perm, shift) uint8 [8, 40] as the library holds them."""
    perm, shift = np.zeros((8, 40), np.uint8), np.zeros((8, 40), np.uint8)
    lib().bbs_tables(_p(perm), _p(shift))
    return perm, shift


def sym_board(g, b):
    return int(lib().bbs_sym_board(int(g), int(b)))


def sym_cell(g, a):
    return int(lib().bbs_sym_cell(int(g), int(a)))


def sym_pieces(g, pw):
    return int(lib().bbs_sym_pieces(int(g), int(pw)))


def sym_anchor(g, piece, a):
    return int(lib().bbs_sym_anchor(int(g), int(piece), int(a)))


def sym_mask_plane(g, piece, plane):
    return int(lib().bbs_sym_mask_plane(int(g), int(piece), int(plane)))


def sym_action(g, pieces_word, action):
    """The image of action slot*64 + anchor under symmetry g, for the state with pieces word ``pieces_word``."""
    slot, a = int(action) >> 6, int(action) & 63
    return slot * 64 + sym_anchor(g, (int(pieces_word) >> (8 * slot)) & 0xFF, a)


def obs_views(board, pieces):
    """Bitboards uint64 [8, n, 4] of the eight views of packed rows (board uint64 [n], pieces uint32 [n])."""
    b = np.ascontiguousarray(board, np.uint64)
    p = np.ascontiguousarray(pieces, np.uint32)
    out = np.zeros((8, b.shape[0], 4), np.uint64)
    lib().bbs_obs_views(_p(b), _p(p), C.c_int64(b.shape[0]), _p(out))
    return out


def step(state, action, trios, cfg=None):
    """One no-auto-reset step of ``state`` (STATE_DTYPE scalar record, copied) on candidate trios uint8 [L, 3].
    Returns (new state, reward f32, terminated, info u32, mask uint64 [3])."""
    from oracle.bb_oracle import REWARD_DEFAULTS, REWARD_KEYS
    c = dict(REWARD_DEFAULTS)
    if cfg:
        c.update(cfg)
    cfg_a = np.array([c[k] for k in REWARD_KEYS], np.float64)
    s = np.array([state], dtype=STATE_DTYPE)
    t = np.ascontiguousarray(trios, np.uint8)
    rew, term, info, mask = np.zeros(1, np.float32), np.zeros(1, np.uint8), np.zeros(1, np.uint32), np.zeros(3, np.uint64)
    lib().bbs_step(_p(s), int(action), _p(cfg_a), _p(t), C.c_int64(t.shape[0]), _p(rew), _p(term), _p(info), _p(mask))
    return s[0], rew[0], int(term[0]), int(info[0]), mask


def sym_rows(g, board, pieces):
    """Per-row symmetry g (int [n]) of packed rows: (board uint64 [n], pieces uint32 [n])."""
    n = len(board)
    ga = np.ascontiguousarray(np.broadcast_to(g, (n,)), np.int32)
    b, p = np.ascontiguousarray(board, np.uint64), np.ascontiguousarray(pieces, np.uint32)
    bo, po = np.zeros(n, np.uint64), np.zeros(n, np.uint32)
    lib().bbs_sym_rows(_p(ga), _p(b), _p(p), C.c_int64(n), _p(bo), _p(po))
    return bo, po


def sym_mask_rows(g, pieces, mask):
    """Mask planes uint64 [3, n] of the transformed rows (``pieces``: the original rows' words)."""
    n = len(pieces)
    ga = np.ascontiguousarray(np.broadcast_to(g, (n,)), np.int32)
    p, m = np.ascontiguousarray(pieces, np.uint32), np.ascontiguousarray(mask, np.uint64)
    out = np.zeros((3, n), np.uint64)
    lib().bbs_sym_mask_rows(_p(ga), _p(p), _p(m), C.c_int64(n), _p(out))
    return out


def sym_action_rows(g, pieces, action):
    """Images int32 [n] of legal actions of the rows (``pieces``: the original rows' words)."""
    n = len(pieces)
    ga = np.ascontiguousarray(np.broadcast_to(g, (n,)), np.int32)
    p, a = np.ascontiguousarray(pieces, np.uint32), np.ascontiguousarray(action, np.int32)
    out = np.zeros(n, np.int32)
    lib().bbs_sym_action_rows(_p(ga), _p(p), _p(a), C.c_int64(n), _p(out))
    return out
