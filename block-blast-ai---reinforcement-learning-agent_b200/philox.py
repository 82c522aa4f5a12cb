"""Host replica of the counter-based RNG streams the CUDA kernels draw from.

The reference draws candidate trios with ``rng.choice(37, size=3, replace=True)`` on a
numpy PCG64 generator (src/game/pieces.py:350-355).  That stream is *replaced* (north_star:
"redraws pieces from a counter-based Philox stream"); parity tests feed the reference /
oracle the trios this module produces.

Philox4x32-10 (Salmon et al., SC'11), one block per event:

    key     = (seed & 0xffffffff, seed >> 32)
    counter = (global_env_id & 0xffffffff, global_env_id >> 32, index, stream)

    stream 0  TRIO    index = the env's draw counter; words 0..2 -> piece ids via
                      mulhi32(word, 37); word 3 unused
    stream 1  POLICY  index = the env's policy-step counter; word 0 picks the k-th valid
                      action, k = mulhi32(word0, n_valid)   (bb_env_step_random)
    stream 2  SAMPLE  categorical sampling in bb_masked_sample: counter =
                      (row & 0xffffffff, row >> 32, call_counter, 2); word 0 -> u in [0,1);
                      the action is the inverse CDF of u * sum(p) taken over the kernel's lane
                      order of the 192 actions (``sample_order()``), a fixed permutation
    stream 3  SAMPLE_VALID  bb_env_sample_valid_actions: index = the caller's call counter;
                      word 0 picks the k-th valid action as in stream 1
    stream 4  LOOKAHEAD  the trios dealt to SUCCESSOR states in bb_env_expand, deliberately
                      NOT the env's own TRIO stream (a planner must not see the trio the env
                      will really be dealt).  Counter = (env_id lo, env_id hi,
                      call_counter << 7 | d, 4 | k << 8): call_counter < 2^25 is the caller's
                      expansion counter, k < 64 the sample index, d < 100 the candidate
                      index within the deal; words 0..2 -> piece ids as in stream 0.  The
                      stream does not depend on the action (common random numbers: every
                      deal of an env with the same k sees the same candidate sequence).

Everything here is numpy on the host; it is documentation-by-code of the device streams and
the generator of candidate-trio fixtures.  It launches nothing and is not a fallback for any
kernel.
"""
import numpy as np

M0 = np.uint64(0xD2511F53)
M1 = np.uint64(0xCD9E8D57)
W0 = 0x9E3779B9
W1 = 0xBB67AE85
MASK32 = np.uint64(0xFFFFFFFF)

STREAM_TRIO = 0
STREAM_POLICY = 1
STREAM_SAMPLE = 2
STREAM_SAMPLE_VALID = 3
STREAM_LOOKAHEAD = 4


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Vectorised Philox4x32-10.  All arguments broadcastable integer arrays; returns a
    tuple of four uint32 arrays."""
    c0, c1, c2, c3 = (np.asarray(x, dtype=np.uint64) & MASK32 for x in (c0, c1, c2, c3))
    c0, c1, c2, c3 = np.broadcast_arrays(c0, c1, c2, c3)
    k0 = int(k0) & 0xFFFFFFFF
    k1 = int(k1) & 0xFFFFFFFF
    for _ in range(10):
        p0 = M0 * c0
        p1 = M1 * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & MASK32
        hi1, lo1 = p1 >> np.uint64(32), p1 & MASK32
        c0, c1, c2, c3 = (hi1 ^ c1 ^ np.uint64(k0)), lo1, (hi0 ^ c3 ^ np.uint64(k1)), lo0
        k0 = (k0 + W0) & 0xFFFFFFFF
        k1 = (k1 + W1) & 0xFFFFFFFF
    return tuple(x.astype(np.uint32) for x in (c0, c1, c2, c3))


def mulhi32(x, n):
    """floor(x * n / 2**32): the u32 -> [0, n) map used on the device (__umulhi)."""
    return ((np.asarray(x, dtype=np.uint64) * np.uint64(n)) >> np.uint64(32)).astype(np.uint32)


def candidate_trios(seed, env_ids, n_draws, first_draw=0):
    """uint8 [len(env_ids), n_draws, 3]: candidate trio number d of global env id e."""
    env_ids = np.asarray(env_ids, dtype=np.uint64).reshape(-1, 1)
    d = (np.arange(n_draws, dtype=np.uint64) + np.uint64(first_draw)).reshape(1, -1)
    w = philox4x32_10(env_ids & MASK32, env_ids >> np.uint64(32), d, STREAM_TRIO,
                      seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    return np.stack([mulhi32(w[k], 37) for k in range(3)], axis=-1).astype(np.uint8)


def lookahead_trios(seed, env_ids, call_counter, k, n_draws):
    """uint8 [len(env_ids), n_draws, 3]: LOOKAHEAD candidates d = 0..n_draws-1 (n_draws <= 100) of
    sample k in expansion call ``call_counter`` for global env ids ``env_ids``."""
    assert 0 <= call_counter < 2 ** 25 and 0 <= k < 64 and 0 < n_draws <= 100
    env_ids = np.asarray(env_ids, dtype=np.uint64).reshape(-1, 1)
    d = np.arange(n_draws, dtype=np.uint64).reshape(1, -1)
    w = philox4x32_10(env_ids & MASK32, env_ids >> np.uint64(32), (np.uint64(call_counter) << np.uint64(7)) | d,
                      STREAM_LOOKAHEAD | (k << 8), seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    return np.stack([mulhi32(w[j], 37) for j in range(3)], axis=-1).astype(np.uint8)


def policy_words(seed, env_ids, steps):
    """uint32 [len(steps), len(env_ids)]: word 0 of the POLICY stream."""
    env_ids = np.asarray(env_ids, dtype=np.uint64).reshape(1, -1)
    s = np.asarray(steps, dtype=np.uint64).reshape(-1, 1)
    w = philox4x32_10(env_ids & MASK32, env_ids >> np.uint64(32), s, STREAM_POLICY,
                      seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    return w[0]


def sample_uniforms(seed, call_counter, n_rows):
    """float32 [n_rows]: u = (word0 >> 8) * 2**-24 of the SAMPLE stream (bb_masked_sample)."""
    rows = np.arange(n_rows, dtype=np.uint64)
    w = philox4x32_10(rows & MASK32, rows >> np.uint64(32), call_counter, STREAM_SAMPLE,
                      seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    return (w[0] >> np.uint32(8)).astype(np.float32) * np.float32(2.0 ** -24)


def sample_order():
    """int64 [192]: the order in which bb_masked_sample accumulates the CDF — lane l of a
    4-lane row group owns actions 16k + 4l + c (k = 0..11, c = 0..3); lanes are scanned in
    order, then k, then c."""
    return np.array([16 * k + 4 * l + c for l in range(4) for k in range(12) for c in range(4)], dtype=np.int64)
