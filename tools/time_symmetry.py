#!/usr/bin/env python3
"""Measure the board-symmetric policies on one GPU, in one run with the card's name, power limit and maximum SM
clock: the eight-view average (K7, PPOConfig.symmetrize) and the canonical frame (K7c, PPOConfig.canonical_frame)
against the plain policy.

Kernels (CUDA events over many launches, outputs larger than L2 at the two large sizes; at 64 states the
numbers are launch overhead): K7a (bb_unpack_obs_sym, n states -> 8n rows) against K2 (bb_unpack_obs) at the
same 8n output rows, and K7b forward / backward (bb_sym_logits_mean[_backward]), f32 and bf16, at 64, 131,072
and 262,144 states, each with its algorithmic HBM bytes and their fraction of the 7.7 TB/s data-sheet figure;
K7c: bb_sym_canonical followed by K2 on the n canonical rows against K2 alone on n rows, and the logit map
forward / backward (bb_sym_logits_canonical[_backward]), f32 and bf16, at the same sizes.

Training shapes (bf16, CUDA graphs; plain, symmetrize and canonical_frame, alternating): rollout time per env step (RolloutRunner:
K7a / K2, CNN, K7b, K3, K1) and PPO update time per minibatch (gather, CNN forward and backward, loss tail, clip,
Adam; GAE and the per-epoch permutation included), each with the peak allocated memory of that phase:
  ref: the reference's schedule, 64 envs x 128 steps, minibatch 2,048, 10 epochs
  cfg4: the config-4 shape of bench.py's ppo leg, 131,072 envs, minibatch 32,768 (8 steps, 1 epoch here)
One JSON line per measurement.

    python tools/time_symmetry.py [--out FILE] [--skip-train]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bbgpu import capi  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def card():
    q = ["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"]
    try:
        smi = subprocess.run(q, capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:                                     # noqa: BLE001
        smi = "nvidia-smi failed: %s" % e
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi}


def event_time_us(fn, reps, warmup=5):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3


def kernels(emit):
    g = torch.Generator("cuda").manual_seed(0)
    for n in (64, 131072, 262144):
        board = torch.randint(-2 ** 62, 2 ** 62, (n,), device="cuda", generator=g)
        ids = torch.randint(0, 37, (n, 3), device="cuda", generator=g)
        pieces = (ids[:, 0] | (ids[:, 1] << 8) | (ids[:, 2] << 16)).to(torch.int32)
        board8 = board.repeat(8)
        pieces8 = pieces.repeat(8)
        reps = 200 if n > 64 else 2000
        for dt in (torch.float32, torch.bfloat16):
            es = 4 if dt == torch.float32 else 2
            name = "f32" if dt == torch.float32 else "bf16"
            obs = torch.empty((8 * n, 4, 8, 8), dtype=dt, device="cuda")
            us_k2 = event_time_us(lambda: capi.unpack_obs(board8, pieces8, None, 8 * n, obs=obs, n=8 * n), reps)
            us_k7a = event_time_us(lambda: capi.unpack_obs_sym(board, pieces, obs, n=n), reps)
            b_k2 = 8 * n * (12 + 256 * es)
            b_k7a = n * 12 + 8 * n * 256 * es
            emit({"kernel": "K2_at_8n_rows", "dtype": name, "states": n, "rows": 8 * n, "us": us_k2, "bytes": b_k2,
                  "hbm_fraction": b_k2 / (us_k2 * 1e-6) / HBM_BYTES_PER_S})
            emit({"kernel": "K7a_unpack_obs_sym", "dtype": name, "states": n, "rows": 8 * n, "us": us_k7a, "bytes": b_k7a,
                  "hbm_fraction": b_k7a / (us_k7a * 1e-6) / HBM_BYTES_PER_S})
            del obs
            logits = torch.randn((8 * n, 192), device="cuda", generator=g).to(dt)
            out = torch.empty((n, 192), dtype=torch.float32, device="cuda")
            grad = torch.empty_like(logits)
            us_f = event_time_us(lambda: capi.sym_logits_mean(logits, pieces, out), reps)
            us_b = event_time_us(lambda: capi.sym_logits_mean_backward(out, pieces, grad), reps)
            b_f = 8 * n * 192 * es + 4 * n + n * 768
            b_b = n * 768 + 4 * n + 8 * n * 192 * es
            emit({"kernel": "K7b_forward", "dtype": name, "states": n, "us": us_f, "bytes": b_f,
                  "hbm_fraction": b_f / (us_f * 1e-6) / HBM_BYTES_PER_S})
            emit({"kernel": "K7b_backward", "dtype": name, "states": n, "us": us_b, "bytes": b_b,
                  "hbm_fraction": b_b / (us_b * 1e-6) / HBM_BYTES_PER_S})
            del logits, out, grad
            # K7c: canonical views + K2 on n rows against K2 alone on n rows; the logit map on n rows
            obs = torch.empty((n, 4, 8, 8), dtype=dt, device="cuda")
            cb, cp = torch.empty_like(board), torch.empty_like(pieces)
            views = torch.empty(n, dtype=torch.uint8, device="cuda")

            def canon_k2():
                capi.sym_canonical(board, pieces, cb, cp, views, n=n)
                capi.unpack_obs(cb, cp, None, n, obs=obs, n=n)
            us_k2n = event_time_us(lambda: capi.unpack_obs(board, pieces, None, n, obs=obs, n=n), reps)
            us_c = event_time_us(lambda: capi.sym_canonical(board, pieces, cb, cp, views, n=n), reps)
            us_ck2 = event_time_us(canon_k2, reps)
            b_k2n = n * (12 + 256 * es)
            b_c = n * (12 + 13)
            b_ck2 = b_c + b_k2n
            emit({"kernel": "K2_at_n_rows", "dtype": name, "states": n, "us": us_k2n, "bytes": b_k2n,
                  "hbm_fraction": b_k2n / (us_k2n * 1e-6) / HBM_BYTES_PER_S})
            emit({"kernel": "K7c_sym_canonical", "dtype": name, "states": n, "us": us_c, "bytes": b_c,
                  "hbm_fraction": b_c / (us_c * 1e-6) / HBM_BYTES_PER_S})
            emit({"kernel": "K7c_sym_canonical_plus_K2", "dtype": name, "states": n, "us": us_ck2, "bytes": b_ck2,
                  "hbm_fraction": b_ck2 / (us_ck2 * 1e-6) / HBM_BYTES_PER_S})
            del obs
            logits = torch.randn((n, 192), device="cuda", generator=g).to(dt)
            out = torch.empty((n, 192), dtype=torch.float32, device="cuda")
            grad = torch.empty_like(logits)
            us_f = event_time_us(lambda: capi.sym_logits_canonical(logits, pieces, views, out), reps)
            us_b = event_time_us(lambda: capi.sym_logits_canonical_backward(out, pieces, views, grad), reps)
            b_f = n * 192 * es + 5 * n + n * 768
            b_b = n * 768 + 5 * n + n * 192 * es
            emit({"kernel": "K7c_map_forward", "dtype": name, "states": n, "us": us_f, "bytes": b_f,
                  "hbm_fraction": b_f / (us_f * 1e-6) / HBM_BYTES_PER_S})
            emit({"kernel": "K7c_map_backward", "dtype": name, "states": n, "us": us_b, "bytes": b_b,
                  "hbm_fraction": b_b / (us_b * 1e-6) / HBM_BYTES_PER_S})
            del logits, out, grad
        torch.cuda.empty_cache()


def train_shape(emit, label, n_envs, T, minibatch, epochs, policy, rollouts, updates):
    from bbgpu.ppo import PPOAgent, PPOConfig
    from bbgpu.rollout import RolloutBuffer
    from bbgpu.train import RolloutRunner
    from bbgpu.vec_env import VectorizedBlockBlastEnv
    dev = torch.device("cuda", 0)
    agent = PPOAgent(PPOConfig(batch_size=minibatch, num_epochs=epochs, precision="bf16", symmetrize=policy == "symmetrize",
                               canonical_frame=policy == "canonical_frame"), dev, seed=1)
    agent.train()
    venv = VectorizedBlockBlastEnv(n_envs, seed=1, output="packed")
    buf = RolloutBuffer(T, n_envs)
    runner = RolloutRunner(venv, agent, buf, use_graph=True)
    for _ in range(2):                                  # eager pass, then capture of both graphs
        lv = runner.run()
        agent.update(buf, lv, use_graph=True)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    for _ in range(rollouts):
        lv = runner.run()
    torch.cuda.synchronize()
    t_roll = (time.perf_counter() - t0) / (rollouts * T)
    peak_roll = torch.cuda.max_memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    for _ in range(updates):
        agent.update(buf, lv, use_graph=True)
    torch.cuda.synchronize()
    n_mb = updates * epochs * (T * n_envs // minibatch)
    t_mb = (time.perf_counter() - t0) / n_mb
    peak_upd = torch.cuda.max_memory_allocated()
    emit({"shape": label, "policy": policy, "envs": n_envs, "rollout_steps": T, "minibatch": minibatch, "epochs": epochs,
          "rollout_step_ms": t_roll * 1e3, "rollout_peak_gb": peak_roll / 1e9, "minibatch_step_ms": t_mb * 1e3,
          "update_peak_gb": peak_upd / 1e9, "rollouts_timed": rollouts, "minibatches_timed": n_mb})
    venv.close()
    del agent, buf, runner, venv
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--skip-train", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_symmetry.py needs a CUDA device")
    torch.cuda.set_device(0)
    f = open(a.out, "w") if a.out else None
    info = card()

    def emit(row):
        line = json.dumps({**row, **info})
        print(line, flush=True)
        if f:
            f.write(line + "\n")
            f.flush()

    kernels(emit)
    if not a.skip_train:
        policies = ("plain", "symmetrize", "canonical_frame")
        for rep in range(2):                                 # alternating arms, twice: the spread is part of the result
            for policy in policies:
                train_shape(emit, "ref", 64, 128, 2048, 10, policy, rollouts=5, updates=3)
            for policy in policies:
                train_shape(emit, "cfg4", 131072, 8, 32768, 1, policy, rollouts=2, updates=2)
    if f:
        f.close()


if __name__ == "__main__":
    main()
