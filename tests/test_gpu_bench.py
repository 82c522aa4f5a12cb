"""bench.py on the GPU: --steps is the number of timed launches, and --dump-outputs writes what the
last of them returned, which the C oracle reproduces from the same seed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DUMP_MAX_ROWS = 65536


@pytest.mark.parametrize("n", [2048, DUMP_MAX_ROWS + 4096])      # every env dumped / a seeded sample of them
def test_bench_dump_is_the_last_timed_launch(tmp_path, n):
    from bbgpu import philox
    from oracle import bb_oracle_c as OC
    M, K, W, P = 2, 5, 3, 8
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(K), "--warmup", str(W),
                        "--envs", str(n), "--batches", str(M), "--preroll", str(P), "--no-cpu", "--no-ppo",
                        "--no-kernels", "--e2e-min-seconds", "0.05", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["steps"] == K and d["gpu_launches"] == K and d["timing"]["launches_timed"] == K
    got = {f[:-4]: np.load(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)}
    assert set(got) == {"env_id", "actions", "rewards", "terminated", "action_mask"}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    # launch k steps batch k % M; batch b has env ids b*n ... and ran the preroll plus its share of the
    # warm-up and timed launches.  Replay it with the random valid-action policy (bench.py's seed 42).
    b = (W + K - 1) % M
    T = P + sum(1 for k in range(W + K) if k % M == b)
    ids = got["env_id"].astype(np.int64)
    rows = min(n, DUMP_MAX_ROWS)
    assert len(ids) == rows and ids[0] >= b * n and ids[-1] < (b + 1) * n and np.all(np.diff(ids) > 0)
    assert all(got[k].shape[0] == rows for k in got)
    sel = np.arange(rows) if n <= DUMP_MAX_ROWS else np.arange(0, rows, 64)   # every dumped row / 1,024 of them
    ids = ids[sel]
    ora = OC.CVecEnv(philox.candidate_trios(42, ids, 512), n_threads=8)
    words = philox.policy_words(42, ids, np.arange(T))
    for t in range(T):
        _, _, m = ora.export()
        bits = np.unpackbits(m.view(np.uint8).reshape(len(ids), 24), axis=1, bitorder="little").astype(np.int64)
        k = philox.mulhi32(words[t], bits.sum(1)).astype(np.int64)
        acts = (np.cumsum(bits, axis=1) <= k[:, None]).sum(axis=1).astype(np.int32)   # the (k+1)-th valid action
        oo = ora.step(acts)
    dense = np.unpackbits(oo["mask"].view(np.uint8).reshape(len(ids), 24), axis=1, bitorder="little")
    assert np.array_equal(got["actions"][sel], acts.astype(np.float32))
    assert np.array_equal(got["rewards"][sel].view(np.uint32), oo["rewards"].view(np.uint32))
    assert np.array_equal(got["terminated"][sel], oo["terminated"].astype(np.float32))
    assert np.array_equal(got["action_mask"][sel], dense.astype(np.float32))
