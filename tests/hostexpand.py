"""ctypes loader for the host build of the one-ply expansion (tests/hostbuild/bb_expand_host.cpp: the
product's rules header compiled for the host, with bb_env_expand's per-item body and the sequential
deal on the LOOKAHEAD stream).  Test infrastructure only.  The library is compiled into a private
temporary directory on first use, so the tests work from a read-only tree."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from hostrules import STATE_DTYPE

_TESTS = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_TESTS, "hostbuild", "bb_expand_host.cpp")
_CSRC = os.path.join(os.path.dirname(_TESTS), "block-blast-ai---reinforcement-learning-agent_b200", "csrc")
_LIB = None

EXPAND_FIELDS = ("action", "reward", "terminated", "info", "board", "pieces")


def lib():
    global _LIB
    if _LIB is None:
        out = tempfile.mkdtemp(prefix="bbx_")
        atexit.register(shutil.rmtree, out, True)
        so = os.path.join(out, "libbbexpand_host.so")
        gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        # the flags of tests/hostbuild/Makefile (no FMA contraction: the float64 reward must be bit-exact)
        subprocess.check_call([gxx, "-O2", "-fPIC", "-ffp-contract=off", "-std=c++17", "-I" + _CSRC, "-x", "c++",
                               "-shared", "-o", so, _SRC], stderr=subprocess.DEVNULL)
        L = C.CDLL(so)
        L.bbx_state_size.restype = C.c_int64
        L.bbx_lookahead_trio.restype = C.c_uint32
        L.bbx_lookahead_trio.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32]
        assert L.bbx_state_size() == STATE_DTYPE.itemsize == 48
        _LIB = L
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def expand(state, seed, call_counter, samples, env_offset=0, cfg=None, capacity=None):
    """bb_env_expand on the host (sequential deal) of the states ``state`` (STATE_DTYPE [n]): dict of
    offsets [n+1], the item arrays and mask [3, capacity]; capacity None = exactly the item count."""
    from oracle.bb_oracle import REWARD_DEFAULTS, REWARD_KEYS
    c = dict(REWARD_DEFAULTS)
    if cfg:
        c.update(cfg)
    cfg_a = np.array([c[k] for k in REWARD_KEYS], np.float64)
    st = np.ascontiguousarray(state, dtype=STATE_DTYPE)
    n = st.shape[0]
    L = lib()

    def call(cap, o):
        L.bbx_expand(_p(st), C.c_int64(n), _p(cfg_a), C.c_uint64(seed), C.c_int64(env_offset), C.c_uint32(call_counter),
                     C.c_int(samples), C.c_int64(cap), _p(o["offsets"]), *[_p(o.get(f)) for f in EXPAND_FIELDS + ("mask",)])

    offsets = np.zeros(n + 1, np.int64)
    if capacity is None:
        call(0, {"offsets": offsets})
        capacity = int(offsets[n])
    out = {"offsets": offsets, "action": np.zeros(capacity, np.int32), "reward": np.zeros(capacity, np.float32),
           "terminated": np.zeros(capacity, np.uint8), "info": np.zeros(capacity, np.uint32),
           "board": np.zeros(capacity, np.uint64), "pieces": np.zeros(capacity, np.uint32),
           "mask": np.zeros((3, capacity), np.uint64)}
    call(capacity, out)
    return out


def lookahead_trio(seed, env_id, call_counter, k, d):
    """LOOKAHEAD candidate d of sample k (bytes 0..2 = piece ids) from the host build."""
    return lib().bbx_lookahead_trio(seed, env_id, call_counter, k, d)
