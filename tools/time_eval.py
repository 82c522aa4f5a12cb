#!/usr/bin/env python3
"""Time the deterministic evaluation with and without live-env compaction on one GPU, in one run with the card's
name, power limit and maximum SM clock.

The agent is a ``tools/train_demo.yaml`` agent trained for ``--train-updates`` updates (or ``--checkpoint``).
For each precision and each episode count the two loops alternate, ``--reps`` timed runs each after one warm-up
run (cuDNN plans every batch shape once per process):
  full     the full-batch loop evaluate ran before compaction, restated below: the network on all n rows at
           every step until the longest episode ends
  compact  ``bbgpu.evaluate.evaluate``: the network on the live rows only (bb_env_observe_live)
Each run reports its wall time (host clock around work that ends in a device synchronise), the network rows
it ran, its steps, the env-steps it issued (steps x n) and the moves actually played (sum of episode lengths),
and whether its per-episode scores equal the other loop's.  One JSON line per run.

    python tools/time_eval.py --out profiles/r3_time_eval_1gpu.jsonl [--checkpoint ck.pt] [--sizes 4096,65536]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bbgpu import capi  # noqa: E402
from bbgpu.evaluate import evaluate  # noqa: E402
from bbgpu.ppo import PPOAgent, PPOConfig  # noqa: E402


def card():
    q = ["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"]
    try:
        smi = subprocess.run(q, capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:                                     # noqa: BLE001
        smi = "nvidia-smi failed: %s" % e
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi}


@torch.no_grad()
def evaluate_full_batch(agent, n, seed, max_steps=10000):
    """The deterministic loop of evaluate before live-env compaction: observe every env, run the network on all n
    rows, step every env, until every episode has ended.  Returns the per-episode scores and lengths."""
    dev = agent.device
    h = capi.EnvHandle(n, seed, 0, None, capi.ENV_NO_AUTO_RESET)
    board = torch.zeros(n, dtype=torch.int64, device=dev)
    pieces = torch.zeros(n, dtype=torch.int32, device=dev)
    mask = torch.zeros((3, n), dtype=torch.int64, device=dev)
    rewards = torch.zeros(n, dtype=torch.float32, device=dev)
    term = torch.zeros(n, dtype=torch.uint8, device=dev)
    done = torch.zeros(n, dtype=torch.bool, device=dev)
    was_training = agent.training
    agent.eval()
    steps = 0
    try:
        while steps < max_steps and not bool(done.all()):
            h.observe(board, pieces, mask)
            act, _, _ = agent.act({"board": board, "pieces": pieces, "mask": mask}, deterministic=True)
            h.step(act, rewards, term, None, None, None, None)
            done |= term.bool()
            steps += 1
        st = h.get_state()
    finally:
        h.close()
        if was_training:
            agent.train()
    return {"scores": st["score"].astype(np.int64), "lengths": st["moves"].astype(np.int64)}


class RowCounter:
    """Counts the network rows of agent.act calls (both loops call it once per step)."""

    def __init__(self, agent):
        self.rows, self.calls, self._act = 0, 0, agent.act
        agent.act = self

    def __call__(self, obs, *a, **k):
        self.rows += int(obs["board"].shape[0])
        self.calls += 1
        return self._act(obs, *a, **k)


def trained_checkpoint(updates, tmp):
    import yaml
    from bbgpu.train import train
    with open(os.path.join(ROOT, "tools", "train_demo.yaml")) as f:
        cfg = yaml.safe_load(f)
    cfg["paths"] = {"checkpoint_dir": os.path.join(tmp, "ck"), "log_dir": os.path.join(tmp, "logs")}
    cfg.setdefault("logging", {})["tensorboard"] = False
    t0 = time.time()
    hist = train(cfg, seed=42, max_updates=updates)
    return os.path.join(tmp, "ck", "final.pt"), {"train_updates": len(hist), "train_wall_s": time.time() - t0,
                                                  "train_avg_score_last": hist[-1]["avg_score"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--checkpoint", default=None)
    ap.add_argument("--train-updates", type=int, default=30)
    ap.add_argument("--sizes", default="4096,65536")
    ap.add_argument("--precisions", default="fp32,bf16")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_eval.py measures on a GPU; none is visible")
    torch.cuda.set_device(0)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    out = open(a.out, "w")

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        out.write(line + "\n")
        out.flush()

    info = card()
    with tempfile.TemporaryDirectory() as tmp:
        if a.checkpoint:
            ck, trained = a.checkpoint, {}
        else:
            ck, trained = trained_checkpoint(a.train_updates, tmp)
        emit({"kind": "setup", **info, "checkpoint": a.checkpoint or "tools/train_demo.yaml", **trained})
        for precision in a.precisions.split(","):
            agent = PPOAgent(PPOConfig(precision=precision))
            agent.load(ck)
            counter = RowCounter(agent)
            for n in [int(x) for x in a.sizes.split(",")]:
                arms = {"full": lambda: evaluate_full_batch(agent, n, a.seed),
                        "compact": lambda: evaluate(agent, n, seed=a.seed)}
                scores = {}
                for rep in range(a.reps + 1):                     # rep 0: warm-up, not reported
                    for arm, fn in arms.items():
                        counter.rows = counter.calls = 0
                        torch.cuda.synchronize()
                        t0 = time.perf_counter()
                        res = fn()
                        torch.cuda.synchronize()
                        wall = time.perf_counter() - t0
                        scores[arm] = res["scores"]
                        if rep == 0:
                            continue
                        other = scores.get("compact" if arm == "full" else "full")
                        emit({"kind": "eval", "arm": arm, "precision": precision, "episodes": n, "rep": rep,
                              "wall_s": wall, "network_rows": counter.rows, "steps": counter.calls,
                              "env_steps": counter.calls * n, "moves": int(res["lengths"].sum()),
                              "mean_score": float(res["scores"].mean()), "mean_length": float(res["lengths"].mean()),
                              "max_length": int(res["lengths"].max()),
                              "scores_equal_other_arm": None if other is None else bool(np.array_equal(other, res["scores"])),
                              "episodes_differing": None if other is None else int((other != res["scores"]).sum()),
                              **info})
    out.close()


if __name__ == "__main__":
    main()
