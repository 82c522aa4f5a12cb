#!/usr/bin/env python3
"""Time bb_env_expand (one-ply successor expansion) on mid-game states, next to K1 in the same run.

For 16,384 / 65,536 / 262,144 envs brought to a steady-state mix of mid-game states by 64 steps of
bb_env_rollout_random, and K = 1 and 4 samples per dealing move: microseconds per call (CUDA events
around the fill call: count + scan + item kernels), items per second, the share of deal items,
algorithmic bytes (48 B state read + 8 B offsets written per env, 49 B written per item) against the
7.7 TB/s HBM data-sheet bandwidth, and the time per item next to K1's time per env-step
(bb_env_step_random, one step per launch, same envs).  Then one evaluate(lookahead=4) step of
1,000 envs, split into expansion, value CNN and the Q reduction.  One JSON line per measurement.

    python tools/time_expand.py [--checkpoint ckpt.pt] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bbgpu import capi  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
FIELDS = ("action", "reward", "terminated", "info", "board", "pieces")
DTYPES = {"action": torch.int32, "reward": torch.float32, "terminated": torch.uint8, "info": torch.int32,
          "board": torch.int64, "pieces": torch.int32}


def card():
    q = ["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"]
    try:
        smi = subprocess.run(q, capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:                                     # noqa: BLE001
        smi = "nvidia-smi failed: %s" % e
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi}


def raw_expand(h, cc, samples, cap, offsets, outs):
    p = capi.ptr
    capi.check(capi.lib().bb_env_expand(h.h, cc, samples, cap, p(offsets), *[p(outs.get(f)) for f in FIELDS + ("mask",)],
                                        capi.current_stream()))


def event_time_us(fn, reps, warmup=3):
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


def kernel_rows(seed, reps):
    rows = []
    for n in (16384, 65536, 262144):
        h = capi.EnvHandle(n, seed)
        h.rollout_random(64)
        offsets = torch.empty(n + 1, dtype=torch.int64, device="cuda")
        for K in (1, 4):
            raw_expand(h, 1, K, 0, offsets, {})
            items = int(offsets[n].item())
            outs = {f: torch.empty(items, dtype=t, device="cuda") for f, t in DTYPES.items()}
            outs["mask"] = torch.empty((3, items), dtype=torch.int64, device="cuda")
            us = event_time_us(lambda: raw_expand(h, 1, K, items, offsets, outs), reps)
            deal = int((((outs["info"].view(torch.int32) >> 11) & 0x7F) > 0).sum().item())
            nbytes = 56 * n + 8 + 49 * items
            rows.append({"what": "bb_env_expand", "envs": n, "samples": K, "us_per_call": round(us, 1),
                         "items": items, "items_per_env": round(items / n, 2), "deal_items": deal,
                         "deal_share": round(deal / max(items, 1), 4), "items_per_s": items / us * 1e6,
                         "ns_per_item": round(us * 1e3 / max(items, 1), 3), "alg_bytes": nbytes,
                         "hbm_share": round(nbytes / (us * 1e-6) / HBM_BYTES_PER_S, 4),
                         "working_set_fits_l2": nbytes < 126e6})
            del outs
        act = torch.empty(n, dtype=torch.int32, device="cuda")
        us_k1 = event_time_us(lambda: h.step_random(1, act), reps)
        rows.append({"what": "K1 step_random(1)", "envs": n, "us_per_launch": round(us_k1, 1),
                     "ns_per_env_step": round(us_k1 * 1e3 / n, 3)})
        h.close()
    return rows


def eval_split(checkpoint, n=1000, K=4, seed=3):
    from bbgpu.evaluate import lookahead_actions
    from bbgpu.ppo import PPOAgent
    agent = PPOAgent()
    if checkpoint:
        agent.load(checkpoint)
    agent.eval()
    h = capi.EnvHandle(n, seed, 0, None, capi.ENV_NO_AUTO_RESET)
    act = torch.zeros(n, dtype=torch.int32, device="cuda")
    rew, term = torch.zeros(n, device="cuda"), torch.zeros(n, dtype=torch.uint8, device="cuda")
    for t in range(8):                                         # a few moves into the game
        h.sample_valid_actions(t, act, None)
        h.step(act, rew, term)
    for _ in range(3):
        lookahead_actions(agent, h, n, 8, K)                   # warm-up (cuDNN algorithm choice, allocator)
    torch.cuda.synchronize()
    reps, t_exp, t_cnn, t_all = 10, 0.0, 0.0, 0.0
    for r in range(reps):
        t0 = time.perf_counter()
        ex = h.expand(8 + r, K)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        v = agent.values({"board": ex["board"], "pieces": ex["pieces"], "mask": ex["mask"]}, chunk=65536)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        lookahead_actions(agent, h, n, 8 + r, K)
        torch.cuda.synchronize()
        t3 = time.perf_counter()
        t_exp += t1 - t0
        t_cnn += t2 - t1
        t_all += t3 - t2
    h.close()
    return {"what": "evaluate(lookahead=%d) step" % K, "envs": n, "items": int(ex["action"].numel()),
            "expand_ms": round(t_exp / reps * 1e3, 3), "value_cnn_ms": round(t_cnn / reps * 1e3, 3),
            "whole_step_ms": round(t_all / reps * 1e3, 3), "trained_checkpoint": bool(checkpoint), "values": int(v.numel())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--checkpoint", default=None, help="agent for the evaluate split (default: untrained network)")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "time_expand.py measures on the GPU"
    rows = [{"what": "card", **card()}] + kernel_rows(1, a.reps) + [eval_split(a.checkpoint)]
    for r in rows:
        print(json.dumps(r), flush=True)
    if a.out:
        with open(a.out, "a") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
