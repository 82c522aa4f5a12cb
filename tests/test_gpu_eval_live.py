"""GPU checks of the live-env observation (bb_env_observe_live) and of the evaluation built on it: the kernel
against bb_env_observe plus torch.nonzero of the game-over bit, its guard bands, the compacted ``evaluate``
against a restated full-batch loop (logits, actions, oracle replay), the in-training held-out evaluation (it
changes nothing of the training run; logs, tags and best_eval.pt round trip) and rank sharding."""
import json
import os
import socket
import sys

import numpy as np
import pytest

from test_gpu_guard_bands import SIZES, Arena

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


@pytest.fixture(autouse=True)
def _numerics(torch):
    """A bf16 PPOAgent turns on cudnn.benchmark for the whole process; these tests also turn TF32 off. Both are
    put back after each test so that later tests see the settings they would see without this file."""
    saved = (torch.backends.cudnn.benchmark, torch.backends.cudnn.deterministic, torch.backends.cudnn.allow_tf32,
             torch.backends.cuda.matmul.allow_tf32)
    yield
    (torch.backends.cudnn.benchmark, torch.backends.cudnn.deterministic, torch.backends.cudnn.allow_tf32,
     torch.backends.cuda.matmul.allow_tf32) = saved


def _over(h):
    return (h.get_state()["aux"] >> 16) & 1


def _observe_live(torch, h, n, stride, fill=0x5A):
    dev = "cuda"
    out = {"board": torch.full((n,), fill, dtype=torch.int64, device=dev),
           "pieces": torch.full((n,), fill, dtype=torch.int32, device=dev),
           "mask": torch.full((3, stride), fill, dtype=torch.int64, device=dev),
           "ids": torch.full((n,), fill, dtype=torch.int32, device=dev),
           "count": torch.full((1,), fill, dtype=torch.int32, device=dev)}
    h.observe_live(out["board"], out["pieces"], out["mask"], out["ids"], out["count"])
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def _patterns(torch, n, seed):
    """(name, handle) with every env live, none live, and mixes from random play without auto-reset"""
    from bbgpu import capi
    yield "all", capi.EnvHandle(n, seed, 0, None, capi.ENV_NO_AUTO_RESET)
    h = capi.EnvHandle(n, seed, 0, None, capi.ENV_NO_AUTO_RESET)
    st = h.get_state()
    st["aux"] |= np.uint32(1 << 16)
    h.set_state(st)
    yield "none", h
    for steps in (6, 25, 80):
        h = capi.EnvHandle(n, seed + steps, 0, None, capi.ENV_NO_AUTO_RESET)
        h.step_random(steps)
        yield "random%d" % steps, h


@pytest.mark.parametrize("n", [1, 31, 33, 127, 129, 1000, 4097, 262144])
def test_observe_live_matches_observe_and_nonzero_of_game_over(torch, n):
    dev = "cuda"
    seen = set()
    for name, h in _patterns(torch, n, 11):
        board = torch.zeros(n, dtype=torch.int64, device=dev)
        pieces = torch.zeros(n, dtype=torch.int32, device=dev)
        mask = torch.zeros((3, n), dtype=torch.int64, device=dev)
        h.observe(board, pieces, mask)
        before = h.get_state()
        live = torch.nonzero(torch.from_numpy(_over(h) == 0)).flatten().numpy()
        m = live.size
        stride = n + 3                                             # a plane stride other than n
        got = _observe_live(torch, h, n, stride)
        assert got["count"][0] == m, name
        assert np.array_equal(got["ids"][:m], live.astype(np.int32)), name
        assert np.array_equal(got["board"][:m], board.cpu().numpy()[live]), name
        assert np.array_equal(got["pieces"][:m], pieces.cpu().numpy()[live]), name
        assert np.array_equal(got["mask"][:, :m], mask.cpu().numpy()[:, live]), name
        # rows >= count and the padding of the mask planes stay untouched
        assert (got["board"][m:] == 0x5A).all() and (got["ids"][m:] == 0x5A).all() and (got["pieces"][m:] == 0x5A).all()
        assert (got["mask"][:, m:] == 0x5A).all()
        again = _observe_live(torch, h, n, stride, fill=-1)
        assert again["count"][0] == m
        for k in ("board", "pieces", "ids"):
            assert np.array_equal(again[k][:m], got[k][:m]), (name, k)
        assert np.array_equal(again["mask"][:, :m], got["mask"][:, :m])
        assert h.get_state().tobytes() == before.tobytes(), name       # state and counters unchanged
        seen.add("mixed" if 0 < m < n else ("all" if m == n else "none"))
        h.close()
    assert seen >= {"all", "none"} and (n < 31 or "mixed" in seen), seen


def test_observe_live_argument_checks_on_a_live_handle(torch):
    from bbgpu import capi
    h = capi.EnvHandle(40, 1, 0, None, capi.ENV_NO_AUTO_RESET)
    b, p, i, c = (torch.zeros(40, dtype=t, device="cuda") for t in (torch.int64, torch.int32, torch.int32, torch.int32))
    with pytest.raises(capi.BBGpuError, match="mask_stride"):
        h.observe_live(b, p, torch.zeros((3, 39), dtype=torch.int64, device="cuda"), i, c)
    with pytest.raises(capi.BBGpuError, match="NULL output"):
        h.observe_live(b, p, None, i, c)
    h.close()
    with pytest.raises(capi.BBGpuError, match="env is NULL"):
        h.observe_live(b, p, torch.zeros((3, 40), dtype=torch.int64, device="cuda"), i, c)


@pytest.mark.parametrize("n", SIZES)
def test_observe_live_stays_inside_its_buffers(torch, n):
    from bbgpu import capi
    A = Arena(torch)
    h = capi.EnvHandle(n, 3, 0, None, capi.ENV_NO_AUTO_RESET)
    h.step_random(12)
    stride = n + 1
    board, pieces = A.alloc((n,), torch.int64), A.alloc((n,), torch.int32)
    mask, ids, count = A.alloc((3, stride), torch.int64), A.alloc((n,), torch.int32), A.alloc((1,), torch.int32)
    h.observe_live(board, pieces, mask, ids, count)
    A.check()
    m = int(count.item())
    assert m == int((_over(h) == 0).sum())
    h.close()


# ----------------------------------------------------------------------------------------------------------
# evaluate: compacted rows against the full batch
# ----------------------------------------------------------------------------------------------------------
def _agent(torch, form, seed=5):
    from bbgpu.ppo import PPOAgent, PPOConfig
    torch.manual_seed(seed)
    return PPOAgent(PPOConfig(symmetrize=form == "symmetrize", canonical_frame=form == "canonical_frame"))


def _replay_through_oracle(res, n, seed):
    from bbgpu import philox
    from oracle import bb_oracle as O
    streams = philox.candidate_trios(seed, np.arange(n), 1024)
    for i in range(n):
        it = iter(streams[i])
        env = O.Env(draw=lambda: next(it))
        total, t, term, info = 0.0, 0, False, None
        while not term:
            _, r, term, _, info = env.step(int(res["actions"][t, i]))
            assert not info["invalid_action"], (i, t)
            total += float(np.float32(r))
            t += 1
        assert info["score"] == res["scores"][i] and info["moves"] == res["lengths"][i] == t, (i, info)
        assert info["lines_cleared"] == res["lines"][i] and info["max_combo"] == res["max_combos"][i]
        assert abs(total - res["rewards_per_episode"][i]) < 1e-4 * max(1.0, abs(total))


@pytest.mark.parametrize("form", ["plain", "symmetrize", "canonical_frame"])
def test_compacted_evaluation_matches_the_full_batch_loop(torch, form):
    """The full-batch loop (every env's row at every step, as evaluate ran it before) is restated here and
    driven with the compacted evaluation's actions.  At every step the live rows' logits (the rows evaluate
    runs) must equal the full batch's logits of the same envs within a band, and the actions must be equal
    wherever the full batch's top-two masked logits are further apart than that band.  fp32 without TF32: the
    two batches differ only in summation order, a few hundred float32 ulps of a row's largest logit at most;
    the band is 2^-12 of it."""
    from bbgpu import capi
    from bbgpu.evaluate import evaluate, live_rows
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = False
    agent = _agent(torch, form)
    n, seed, dev = 48, 9, "cuda"
    res = evaluate(agent, num_episodes=n, seed=seed, return_actions=True)
    assert res["finished"] == n and agent.training
    acts = torch.from_numpy(res["actions"]).to(dev)
    h = capi.EnvHandle(n, seed, 0, None, capi.ENV_NO_AUTO_RESET)
    board = torch.zeros(n, dtype=torch.int64, device=dev)
    pieces = torch.zeros(n, dtype=torch.int32, device=dev)
    mask = torch.zeros((3, n), dtype=torch.int64, device=dev)
    lb, lp, lm = torch.zeros_like(board), torch.zeros_like(pieces), torch.zeros_like(mask)
    ids, count = torch.zeros(n, dtype=torch.int32, device=dev), torch.zeros(1, dtype=torch.int32, device=dev)
    rew, term = torch.zeros(n, device=dev), torch.zeros(n, dtype=torch.uint8, device=dev)
    bit = 1 << torch.arange(64, device=dev, dtype=torch.int64)
    agent.eval()
    in_band = 0
    try:
        for t in range(acts.shape[0]):
            h.observe(board, pieces, mask)
            full = {"board": board, "pieces": pieces, "mask": mask}
            lf, _, _ = agent._policy(full)
            a_full, _, _ = agent.act(full, deterministic=True)
            h.observe_live(lb, lp, lm, ids, count)
            m = int(count.item())
            assert m > 0
            rows = live_rows(m, n)
            ll, _, _ = agent._policy({"board": lb[:rows], "pieces": lp[:rows], "mask": lm[:, :rows]})
            idx = ids[:m].long()
            want = lf[idx].float()
            band = 2.0 ** -12 * want.abs().amax(1, keepdim=True).clamp(min=1.0)
            assert ((ll[:m].float() - want).abs() <= band).all(), (t, float((ll[:m].float() - want).abs().max()))
            valid = ((mask[:, idx].unsqueeze(-1) & bit) != 0).permute(1, 0, 2).reshape(m, 192)
            top2 = torch.where(valid, want, torch.full_like(want, float("-inf"))).topk(2, dim=1).values
            gap = top2[:, 0] - top2[:, 1]                                    # inf: one valid action
            clear = gap > band[:, 0]
            assert torch.equal(acts[t, idx][clear], a_full[idx][clear]), t
            in_band += int((~clear).any())
            h.step(acts[t], rew, term, None, None, None, None)
        st = h.get_state()
    finally:
        h.close()
        agent.train()
    print("%s: %d of %d steps have a live env whose top-two logits lie inside the band" % (form, in_band, acts.shape[0]))
    assert np.array_equal(st["score"], res["scores"]) and (((st["aux"] >> 16) & 1) == 1).all()
    _replay_through_oracle(res, n, seed)


def test_live_rows_rounds_up_to_four_sizes_per_octave():
    from bbgpu.evaluate import live_rows
    assert [live_rows(m, 10 ** 6) for m in (1, 5, 8, 9, 1000, 1025)] == [1, 5, 8, 10, 1024, 1280]
    assert live_rows(1000, 1003) == 1003 and live_rows(7, 7) == 7
    sizes = {live_rows(m, 1 << 20) for m in range(1, 1 << 16)}
    assert len(sizes) <= 4 * 16 + 4 and all(m <= live_rows(m, 1 << 20) < m * 1.25 + 1 for m in range(1, 5000))


# ----------------------------------------------------------------------------------------------------------
# held-out evaluation inside train()
# ----------------------------------------------------------------------------------------------------------
def _cfg(tmp, precision, **ours):
    return {"training": {"num_envs": 64, "batch_size": 256, "rollout_steps": 8, "total_timesteps": 10 ** 9},
            "ppo": {"num_epochs": 2},
            "logging": {"log_interval": 1, "save_interval": 10 ** 6, "tensorboard": True},
            "paths": {"checkpoint_dir": os.path.join(tmp, "ck"), "log_dir": os.path.join(tmp, "logs")},
            "b200": dict({"precision": precision}, **ours)}


def _snapshot(torch, agent, vec_env, buffer, runner):
    net = agent.network
    opt = agent.optimizer.state_dict()
    return {"net": {k: v.detach().clone() for k, v in net.state_dict().items()},
            "opt": [{k: (v.detach().clone() if torch.is_tensor(v) else v) for k, v in s.items()} for s in opt["state"].values()],
            "calls": net.sample_calls, "rng_cpu": torch.get_rng_state(), "rng_cuda": torch.cuda.get_rng_state(),
            "env": vec_env._handle.get_state().tobytes(),
            "env_tensors": {k: v.clone() for k, v in vars(vec_env).items() if torch.is_tensor(v)},
            "buffer": {k: v.clone() for k, v in vars(buffer).items() if torch.is_tensor(v)},
            "graphs": (runner.graph, agent._graph and agent._graph["graph"], agent._graph and agent._graph["key"]),
            "mode": (agent.training, net.training, agent.config.symmetrize, agent.config.canonical_frame)}


def _same(torch, a, b):
    if isinstance(a, dict):
        return a.keys() == b.keys() and all(_same(torch, a[k], b[k]) for k in a)
    if isinstance(a, (list, tuple)):
        return len(a) == len(b) and all(_same(torch, x, y) for x, y in zip(a, b))
    if torch.is_tensor(a):
        return a.dtype == b.dtype and a.shape == b.shape and torch.equal(a, b)
    return a is b or a == b


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_in_training_evaluation_leaves_training_untouched(torch, tmp_path, monkeypatch, precision):
    """Snapshots of everything an update reads or writes, taken around each in-training evaluation of a
    graph-captured run, are identical; and a run with evaluations ends with the parameters of a run without
    them, when two runs without them agree bit for bit."""
    import inspect
    from bbgpu import train as T
    torch.backends.cudnn.deterministic = True
    real = T.evaluate_held_out
    checked = []

    def wrapped(agent, ev, reward_config, device):
        f = inspect.currentframe().f_back.f_locals                 # train()'s own objects
        assert f["runner"].graph is not None and agent._graph is not None      # both graphs are captured
        before = _snapshot(torch, agent, f["vec_env"], f["buffer"], f["runner"])
        out = real(agent, ev, reward_config, device)
        after = _snapshot(torch, agent, f["vec_env"], f["buffer"], f["runner"])
        assert _same(torch, before, after)
        checked.append(out)
        return out

    monkeypatch.setattr(T, "evaluate_held_out", wrapped)
    params = []
    for k, ours in enumerate([{}, {}, {"eval_interval": 2, "eval_episodes": 64}]):
        hist = T.train(_cfg(str(tmp_path / str(k)), precision, **ours), seed=3, max_updates=4)
        assert len(hist) == 4
        params.append({n: p.detach().clone() for n, p in torch.load(str(tmp_path / str(k) / "ck" / "final.pt"),
                                                                    weights_only=True)["network_state_dict"].items()})
    assert len(checked) == 2 and all(r["eval_finished"] == 64 for r in checked)
    if not _same(torch, params[0], params[1]):
        pytest.skip("two %s runs without evaluation differ in their parameters here" % precision)
    assert _same(torch, params[0], params[2])


def test_evaluation_rows_tags_and_best_eval_checkpoint_round_trip(torch, tmp_path):
    from bbgpu.evaluate import evaluate
    from bbgpu.logger import EVAL_KEYS, tensorboard_tags
    from bbgpu.ppo import PPOAgent
    from bbgpu.train import train
    torch.backends.cudnn.benchmark = False
    cfg = _cfg(str(tmp_path), "fp32", eval_interval=2, eval_episodes=96, eval_seed=77)
    hist = train(cfg, seed=4, max_updates=3)
    logs = [f for f in os.listdir(str(tmp_path / "logs")) if f.endswith(".jsonl")]
    rows = [json.loads(l) for l in open(str(tmp_path / "logs" / logs[0]))]
    assert len(rows) == 3
    assert not any(k in rows[0] for k in EVAL_KEYS)
    for r in rows[1:]:                                       # update 2, and update 3 (training stops)
        assert all(k in r for k in EVAL_KEYS) and r["eval_finished"] == 96
        assert {"evaluation/" + k[5:] for k in EVAL_KEYS} <= set(tensorboard_tags(r))
    assert [r.get("eval_mean_score") for r in rows] == [h.get("eval_mean_score") for h in hist]
    if os.path.isdir(str(tmp_path / "logs" / "ppo_b200")):   # TensorBoard installed: its event file got written
        assert any(f.startswith("events.") for _, _, fs in os.walk(str(tmp_path / "logs")) for f in fs)
    best = max(r["eval_mean_score"] for r in rows[1:])
    agent = PPOAgent()
    agent.load(str(tmp_path / "ck" / "best_eval.pt"))
    res = evaluate(agent, 96, seed=77)
    assert res["mean_score"] == best


def test_sharded_evaluations_start_from_the_single_evaluations_states(torch, monkeypatch):
    from bbgpu import capi
    from bbgpu import evaluate as E
    from bbgpu.train import eval_stats, eval_sums
    starts = []

    class Recording(capi.EnvHandle):
        def __init__(self, *a, **k):
            super().__init__(*a, **k)
            starts.append(self.get_state())

    monkeypatch.setattr(capi, "EnvHandle", Recording)
    agent = _agent(torch, "plain", seed=8)
    n, seed = 96, 21
    E.evaluate(agent, n, seed=seed)
    halves = [E.evaluate(agent, n // 2, seed=seed, global_env_offset=off) for off in (0, n // 2)]
    assert np.concatenate(starts[1:]).tobytes() == starts[0].tobytes()
    parts = [eval_sums(r) for r in halves]
    got = eval_stats([a + b for a, b in zip(*[p[0] for p in parts])], [max(a, b) for a, b in zip(*[p[1] for p in parts])], 0.0)
    s = np.concatenate([r["scores"] for r in halves])
    ln = np.concatenate([r["lengths"] for r in halves])
    assert got["eval_mean_score"] == float(s.mean()) and got["eval_mean_length"] == float(ln.mean())
    assert got["eval_max_score"] == s.max() and got["eval_min_score"] == s.min() and got["eval_finished"] == n
    assert abs(got["eval_std_score"] - float(s.std())) <= 1e-9 * max(float(s.std()), 1.0)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gloo_train_worker(rank, world, port, cfg, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK="0")                           # both ranks on the one GPU
    sys.path.insert(0, ROOT)
    import torch
    from bbgpu import dist
    from bbgpu.train import train
    torch.backends.cudnn.benchmark = False
    dist.init("gloo")
    hist = train(cfg, seed=6, max_updates=1)
    out.put((rank, {k: v for k, v in hist[-1].items() if k.startswith("eval_")}))
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()


def test_two_rank_gloo_job_evaluates_the_games_of_one_rank(torch, tmp_path):
    """Two ranks (gloo, one GPU) evaluate their halves of the games with rank 0's network; the logged result is
    what one process computes for the same network over the same games, shard by shard."""
    import torch.multiprocessing as mp
    from bbgpu.evaluate import evaluate
    from bbgpu.ppo import PPOAgent
    from bbgpu.train import eval_stats, eval_sums
    cfg = _cfg(str(tmp_path), "fp32", eval_interval=1, eval_episodes=64, eval_seed=5, cuda_graph=False)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_train_worker, args=(r, 2, port, cfg, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=600) for _ in range(2))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    (_, e0), (_, e1) = res
    assert e0 == e1 and e0["eval_finished"] == 64
    torch.backends.cudnn.benchmark = False
    agent = PPOAgent()
    agent.load(str(tmp_path / "ck" / "final.pt"))
    parts = [eval_sums(evaluate(agent, 32, seed=5, global_env_offset=off)) for off in (0, 32)]
    want = eval_stats([a + b for a, b in zip(parts[0][0], parts[1][0])],
                      [max(a, b) for a, b in zip(parts[0][1], parts[1][1])], 0.0)
    for k in ("eval_mean_score", "eval_std_score", "eval_max_score", "eval_min_score", "eval_mean_length", "eval_finished"):
        assert e0[k] == want[k], (k, e0[k], want[k])
