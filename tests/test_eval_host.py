"""CPU checks of the held-out evaluation plumbing: the C ABI's argument checks of bb_env_observe_live, the
``b200.eval_*`` settings of train.py, the reduction of shard results, and the ``evaluation/*`` TensorBoard tags."""
import ctypes as C

import numpy as np
import pytest


@pytest.fixture(scope="module")
def lib():
    import bbgpu.build as b
    b.build()
    from bbgpu import capi
    return capi.lib()


def test_c_abi_rejects_bad_arguments_of_observe_live(lib):
    one = C.c_void_p(16)                       # never dereferenced: every call fails its NULL checks first
    f = lib.bb_env_observe_live
    assert f(None, one, one, one, 8, one, one, None) == -1 and b"env is NULL" in lib.bb_last_error()
    for k in range(5):
        outs = [one] * 5
        outs[k] = None
        board, pieces, mask, ids, count = outs
        assert f(one, board, pieces, mask, 8, ids, count, None) == -1, k
        assert b"NULL output" in lib.bb_last_error(), k


def test_eval_settings_defaults_and_divisibility():
    from bbgpu.train import eval_settings
    assert eval_settings({}, 1, 42) is None
    assert eval_settings({"eval_interval": 0, "eval_episodes": 7}, 8, 42) is None
    ev = eval_settings({"eval_interval": 5}, 8, 42)
    assert ev == {"interval": 5, "episodes": 1000, "seed": 43, "lookahead": 0, "max_steps": 10000}
    ev = eval_settings({"eval_interval": 1, "eval_episodes": 96, "eval_seed": 7, "eval_lookahead": 2,
                        "eval_max_steps": 50}, 4, 0)
    assert ev == {"interval": 1, "episodes": 96, "seed": 7, "lookahead": 2, "max_steps": 50}
    with pytest.raises(ValueError, match="divisible by the number of GPUs"):
        eval_settings({"eval_interval": 1, "eval_episodes": 1001}, 2, 0)
    with pytest.raises(ValueError):
        eval_settings({"eval_interval": 1, "eval_episodes": 0}, 1, 0)
    with pytest.raises(ValueError):
        eval_settings({"eval_interval": -1}, 1, 0)


def test_train_refuses_indivisible_eval_episodes_before_touching_a_device(monkeypatch):
    """train() raises at config validation, like it does for num_envs; the CUDA calls before it are stubbed."""
    import torch
    from bbgpu import train as T
    monkeypatch.setattr(T.dist, "init", lambda: (0, 3, 0))
    monkeypatch.setattr(torch.cuda, "set_device", lambda d: None)
    monkeypatch.setattr(T, "set_seed", lambda s: None)
    cfg = {"training": {"num_envs": 96}, "b200": {"eval_interval": 1, "eval_episodes": 100},
           "paths": {"checkpoint_dir": "/nonexistent/ck", "log_dir": "/nonexistent/logs"}}
    monkeypatch.setattr(T.os, "makedirs", lambda *a, **k: None)
    with pytest.raises(ValueError, match="eval_episodes"):
        T.train(cfg)


def test_shard_reduction_equals_statistics_of_the_concatenated_episodes():
    from bbgpu.train import eval_stats, eval_sums
    rs = np.random.RandomState(0)
    shards = [{"scores": rs.randint(0, 5000, 37), "lengths": rs.randint(1, 300, 37), "finished": 37 - k}
              for k in range(4)]
    parts = [eval_sums(r) for r in shards]
    sums = [sum(p[0][j] for p in parts) for j in range(5)]
    maxes = [max(p[1][j] for p in parts) for j in range(2)]
    got = eval_stats(sums, maxes, 1.5)
    s = np.concatenate([r["scores"] for r in shards])
    ln = np.concatenate([r["lengths"] for r in shards])
    assert got["eval_mean_score"] == float(s.mean()) and got["eval_mean_length"] == float(ln.mean())
    assert got["eval_max_score"] == s.max() and got["eval_min_score"] == s.min()
    assert got["eval_finished"] == 37 * 4 - 6 and got["eval_wall_s"] == 1.5
    assert abs(got["eval_std_score"] - float(s.std())) <= 1e-9 * float(s.std())


def test_tensorboard_tags_of_evaluation_rows():
    from bbgpu.logger import EVAL_KEYS, tensorboard_tags
    base = {"avg_score": 1.0, "max_score": 2, "best_score": 1.0, "avg_length": 3.0, "fps": 4.0}
    assert not any(k.startswith("evaluation/") for k in tensorboard_tags(base))
    row = dict(base, **{k: float(i) for i, k in enumerate(EVAL_KEYS)})
    tags = tensorboard_tags(row)
    assert {k for k in tags if k.startswith("evaluation/")} == {
        "evaluation/mean_score", "evaluation/std_score", "evaluation/max_score", "evaluation/min_score",
        "evaluation/mean_length", "evaluation/finished", "evaluation/wall_s"}
    assert tags["evaluation/mean_score"] == 0.0 and tags["evaluation/wall_s"] == 6.0
