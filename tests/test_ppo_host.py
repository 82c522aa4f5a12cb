"""CPU-only tests of the host-side PPO plumbing: network layout, mask packing, env sharding,
and the multi-rank logic (flat gradient bucket, scalar all-reduce) on a world_size-2 gloo group."""
import copy
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_network_layout_matches_reference_spec():
    from bbgpu.network import BlockBlastNetwork
    net = BlockBlastNetwork()
    assert sum(p.numel() for p in net.parameters()) == 5_290_113        # SURVEY.md §2 C1
    keys = list(net.state_dict().keys())
    assert keys[0] == "conv_encoder.0.weight" and "conv_encoder.6.conv1.weight" in keys
    assert "fc_encoder.0.weight" in keys and "policy_head.2.bias" in keys and "value_head.2.weight" in keys
    assert net.state_dict()["fc_encoder.0.weight"].shape == (512, 8192)
    assert net.state_dict()["policy_head.2.weight"].shape == (192, 256)
    logits, value = net.forward(torch.zeros(2, 8, 8), torch.zeros(2, 3, 8, 8), torch.ones(2, 192))
    assert logits.shape == (2, 192) and value.shape == (2,)
    m = torch.ones(2, 192)
    m[:, 5] = 0
    logits, _ = net.forward(torch.zeros(2, 8, 8), torch.zeros(2, 3, 8, 8), m)
    assert torch.isinf(logits[:, 5]).all() and torch.isfinite(logits[:, 6]).all()


def test_network_is_state_dict_compatible_with_reference():
    """Against what the reference's own network computed (tests/golden/policy_golden.npz, make_golden.py
    record_policy): its BlockBlastNetwork() after torch.manual_seed(0), eval mode, on the observations of its
    VectorizedBlockBlastEnv(64, seed=5) after 7 sample_valid_actions steps under numpy seed 11, which the oracle
    rebuilds.  Equal logits from the same seed mean that every parameter up to the policy head is created in the
    reference's order, with its shape and its initialisation, so the state_dicts load into each other."""
    from oracle import bb_oracle as O
    from bbgpu.network import BlockBlastNetwork
    g = np.load(os.path.join(ROOT, "tests", "golden", "policy_golden.npz"))
    vec = O.VecEnv([O.Env(seed=5 + i, rng_factory=O.numpy_rng_factory) for i in range(64)])
    obs, _ = vec.reset()
    rs = np.random.RandomState(11)
    for _ in range(7):
        obs, *_ = vec.step(vec.sample_valid_actions(rs))
    assert np.array_equal(obs["action_mask"].astype(np.uint8), g["mask"])
    torch.manual_seed(0)
    net = BlockBlastNetwork()
    net.eval()
    b, p, m = torch.from_numpy(obs["board"]), torch.from_numpy(obs["pieces"]), torch.from_numpy(g["mask"]).float()
    with torch.no_grad():
        raw, _ = net.forward(b, p, None)
        np.testing.assert_allclose(raw.numpy() * 3.0, g["logits"], rtol=1e-5, atol=1e-5)   # recorded: raw x 3
        lm, _ = net.forward(b, p, m)
        assert torch.equal(torch.isinf(lm), m == 0) and torch.equal(lm[m == 1], raw[m == 1])
        assert np.array_equal(lm.argmax(1).numpy(), g["argmax"])
        # differentiable evaluation path == the reference's get_action_and_value for the recorded actions, on the
        # recorded (x 3) logits: scale the policy head's output layer by 3
        net.policy_head[2].weight.mul_(3.0)
        net.policy_head[2].bias.mul_(3.0)
        _, lp, en, _ = net.evaluate_actions(torch.cat([b.unsqueeze(1), p], 1), m, torch.from_numpy(g["actions"]))
    np.testing.assert_allclose(lp.numpy(), g["log_prob"], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(en.numpy(), g["entropy"], rtol=1e-5, atol=1e-5)


def test_mask_plane_packing():
    from bbgpu.network import _pack_mask_planes
    rs = np.random.RandomState(0)
    m = rs.rand(7, 192) < 0.4
    m[0] = True
    pl = _pack_mask_planes(torch.from_numpy(m)).numpy().view(np.uint64)
    want = np.array([[sum(1 << k for k in range(64) if m[i, p * 64 + k]) for i in range(7)] for p in range(3)], dtype=np.uint64)
    assert np.array_equal(pl, want)


def test_env_sharding_covers_all_envs_once():
    from bbgpu import dist
    for total, world in ((1_048_576, 8), (64, 2), (10, 4), (7, 8)):
        got = [dist.shard(total, r, world) for r in range(world)]
        assert sum(n for _, n in got) == total
        pos = 0
        for off, n in got:
            assert off == pos
            pos += n
    assert dist.shard(1_048_576, 3, 8) == (393216, 131072)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gloo_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    sys.path.insert(0, ROOT)
    from bbgpu import dist
    r, w, _ = dist.init("gloo")
    assert (r, w) == (rank, world) and dist.world_size() == world
    torch.manual_seed(100 + rank)
    lin = torch.nn.Sequential(torch.nn.Linear(5, 3), torch.nn.Linear(3, 2))
    dist.broadcast_module(lin)                                # everyone now has rank 0's weights
    w0 = torch.cat([p.detach().flatten() for p in lin.parameters()])
    bucket = dist.FlatGradBucket(lin.parameters())
    x = torch.full((4, 5), float(rank + 1))
    bucket.zero()
    lin(x).sum().backward()
    local = bucket.flat.clone()
    bucket.all_reduce_mean()                                  # C1: one flat all-reduce, averaged
    tot = dist.all_reduce_scalars([rank + 1.0, 10.0 * (rank + 1)], device="cpu")
    mx = dist.all_reduce_scalars([rank + 1.0], op="max", device="cpu")
    # two-slice mode: the last Linear's gradients (early slice) are reduced from a post-accumulate hook while
    # backward is still running, the rest afterwards; two consecutive steps give the plain mean both times
    lin2 = torch.nn.Sequential(torch.nn.Linear(5, 3), torch.nn.Linear(3, 2))
    dist.broadcast_module(lin2)
    # the local gradients come from a plain copy: the bucket's early slice may already be mid-reduction
    # (in place, on gloo's thread) when backward returns
    plain = copy.deepcopy(lin2)
    b2 = dist.FlatGradBucket(lin2.parameters(), early_from=2)
    early = []
    for step in range(2):
        b2.zero()
        (lin2(x * (step + 1)).sum() * (rank + 2)).backward()
        fired = b2._work is not None
        b2.all_reduce_mean()
        plain.zero_grad()
        (plain(x * (step + 1)).sum() * (rank + 2)).backward()
        loc2 = torch.cat([p.grad.flatten() for p in plain.parameters()])
        early.append((fired, loc2.tolist(), b2.flat.tolist()))
    out.put((rank, w0.tolist(), local.tolist(), bucket.flat.tolist(), tot, mx, dist.shard(9), early))
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()


def test_two_rank_gloo_gradient_bucket_and_scalars():
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gloo_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    (r0, w0, l0, a0, t0, m0, s0, e0), (r1, w1, l1, a1, t1, m1, s1, e1) = res
    for (f0, loc0, red0), (f1, loc1, red1) in zip(e0, e1):       # overlapped two-slice reduction
        assert f0 and f1                                        # the early slice went out from the hook
        assert np.allclose(red0, red1) and np.allclose(red0, (np.array(loc0) + np.array(loc1)) / 2) and loc0 != loc1
    assert w0 == w1                                            # broadcast worked
    assert np.allclose(a0, a1) and np.allclose(a0, (np.array(l0) + np.array(l1)) / 2)
    assert l0 != l1
    assert t0 == t1 == [3.0, 30.0] and m0 == m1 == [2.0]
    assert s0 == (0, 5) and s1 == (5, 4)


# ---------------------------------------------------------------------------------------------
# metrics surface (SURVEY §8f item 3) and GameState serialisation (item 4): host-only parts
# ---------------------------------------------------------------------------------------------
def test_logger_writes_reference_keys_and_summary(tmp_path):
    import json
    from bbgpu.logger import Logger, MetricsTracker, TensorBoardLogger, tensorboard_tags
    lg = Logger(str(tmp_path), name="unit")
    rows = []
    for k in range(1, 4):
        row = {"step": 1000 * k, "fps": 10.0 * k, "avg_score": np.float32(5 * k), "max_score": np.int64(9 * k),
               "best_score": 5.0 * k, "avg_length": 12.5, "policy_loss": -0.01, "value_loss": 0.5, "entropy": 3.0,
               "total_loss": 0.2, "approx_kl": 0.001, "clip_fraction": 0.05}
        rows.append(lg.log(row, 1000 * k))
    lines = [json.loads(l) for l in open(lg.log_file)]
    assert len(lines) == 3 and lines[-1]["step"] == 3000 and lines[1]["avg_score"] == 10.0
    # keys of scripts/train.py:231-243 + the record fields of src/utils/logger.py:66-71
    for key in ("step", "time", "timestamp", "fps", "avg_score", "max_score", "best_score", "avg_length",
                "policy_loss", "value_loss", "entropy", "approx_kl", "clip_fraction"):
        assert key in lines[0]
    assert lg.get_mean("fps") == 20.0 and lg.get_recent("fps", 2) == [20.0, 30.0]
    summ = json.load(open(lg.save_summary()))
    assert summ["total_steps"] == 3000 and summ["metrics"]["fps"] == {"mean": 20.0, "std": float(np.std([10, 20, 30])),
                                                                     "min": 10.0, "max": 30.0, "last": 30.0}
    tags = tensorboard_tags(rows[0])
    assert set(tags) == {"performance/avg_score", "performance/max_score", "performance/best_score",
                         "performance/avg_length", "performance/fps", "training/policy_loss", "training/value_loss",
                         "training/entropy", "training/approx_kl", "training/clip_fraction"}
    tb = TensorBoardLogger(str(tmp_path), name="tb")
    tb.log_metrics(tags, 1000)
    tb.log_scalars("group", {"a": 1.0, "b": 2.0}, 1000)
    tb.close()
    assert not tb.enabled or any(f.startswith("events.") for _, _, fs in __import__("os").walk(str(tmp_path / "tb")) for f in fs)
    tr = MetricsTracker(window_size=3)
    for v in (1, 2, 3, 4):
        tr.add("episode_score", v)
    tr.add_many("episode_length", np.array([7, 9]))
    assert tr.get_mean("episode_score") == 3.0 and tr.get_max("episode_score") == 4.0 and tr.get_min("episode_score") == 2.0
    assert tr.get_last("episode_length") == 9.0 and tr.get_mean("missing") == 0.0
    assert set(tr.get_all_summaries()) == {"episode_score", "episode_length"}
    tr.reset()
    assert tr.get_mean("episode_score") == 0.0


def test_game_state_dict_round_trip():
    import json
    from bbgpu.vec_env import GameState
    board = np.zeros((8, 8), np.int8)
    board[2, 3] = board[7, 7] = 1
    gs = GameState(board=board, current_pieces=[3, 17, 36], pieces_used=[False, True, False], score=123,
                   combo_count=2, moves_made=9, status="playing")
    d = json.loads(json.dumps(gs.to_dict()))
    assert set(d) == {"board", "current_pieces", "pieces_used", "score", "combo_count", "moves_made", "status"}
    back = GameState.from_dict(d)
    assert np.array_equal(back.board, board) and back.board.dtype == np.int8
    assert (back.current_pieces, back.pieces_used, back.score, back.combo_count, back.moves_made, back.status) == \
        ([3, 17, 36], [False, True, False], 123, 2, 9, "playing")


def test_flat_bucket_clip_matches_torch_clip_grad_norm():
    import torch
    from bbgpu.dist import FlatGradBucket
    torch.manual_seed(0)
    for scale in (0.01, 30.0):                      # below and above the threshold
        lin = torch.nn.Sequential(torch.nn.Linear(7, 5), torch.nn.Linear(5, 3))
        ref = torch.nn.Sequential(torch.nn.Linear(7, 5), torch.nn.Linear(5, 3))
        ref.load_state_dict(lin.state_dict())
        bucket = FlatGradBucket(lin.parameters())
        x = torch.randn(11, 7) * scale
        lin(x).pow(2).sum().backward()
        ref(x).pow(2).sum().backward()
        n1 = bucket.clip_grad_norm_(0.5)
        n2 = torch.nn.utils.clip_grad_norm_(ref.parameters(), 0.5)
        torch.testing.assert_close(n1, n2)
        for a, b in zip(lin.parameters(), ref.parameters()):
            assert a.grad.data_ptr() >= bucket.flat.data_ptr()          # still views of the bucket
            torch.testing.assert_close(a.grad, b.grad)


def test_cpulist_parser_and_numa_binding_never_raises():
    """dist.pin_to_gpu_numa is best effort: on a box without NVML / sysfs topology it reports why and
    leaves the affinity alone."""
    import os
    from bbgpu import dist
    assert dist._parse_cpulist("0-3,8,10-11\n") == [0, 1, 2, 3, 8, 10, 11]
    assert dist._parse_cpulist("") == []
    before = os.sched_getaffinity(0)
    info = dist.pin_to_gpu_numa(0, 1)
    assert isinstance(info, dict) and ("error" in info or info.get("cpus"))
    if "error" in info:
        assert os.sched_getaffinity(0) == before
    else:
        os.sched_setaffinity(0, before)


def test_shard_is_even_and_contiguous():
    from bbgpu import dist
    offs = [dist.shard(512, r, 8) for r in range(8)]
    assert offs == [(64 * r, 64) for r in range(8)]
    assert dist.shard(9, 0, 2) == (0, 5) and dist.shard(9, 1, 2) == (5, 4)     # train.py refuses such a job


def test_bench_reference_arm_prints_one_contract_line():
    """bench.py --impl reference (the CPU arm of the driver's comparison) runs without a GPU and prints exactly
    one JSON line with the contract's keys; kind says whether the real reference (oracle/_ref) or the port ran."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "env_steps_per_sec" and d["value"] > 100
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    have_copy = os.path.isdir(os.path.join(root, "oracle", "_ref", "src", "environment"))
    assert d["cpu_baseline"]["kind"] == ("reference" if have_copy else "port")
