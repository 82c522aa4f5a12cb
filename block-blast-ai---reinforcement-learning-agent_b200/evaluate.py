"""Batched evaluation of a trained agent — the reference's ``scripts/evaluate.py:23-90``
(one env, ``deterministic=True`` argmax rollouts) run for many episodes at once on the GPU.

Each of ``num_episodes`` envs plays exactly one episode (``BB_ENV_NO_AUTO_RESET``: a finished env
stays GAME_OVER and its further steps are no-ops), so the returned statistics are per-episode
like the reference's: scores, lengths, lines cleared, max combo.

    python -m bbgpu.evaluate --checkpoint checkpoints/best.pt --episodes 1000

``--lookahead K`` (K >= 1) replaces the argmax policy by a one-ply value look-ahead: every legal move
of every env is expanded on the GPU (``bb_env_expand``; a move that places the last piece is dealt K
sampled trios from the look-ahead stream, never the env's own), the successors are scored by the value
head, and each env plays the move with the highest mean ``reward + gamma * (1 - terminated) * V``.
"""
import argparse
import json

import numpy as np
import torch

from . import capi
from .ppo import PPOAgent


@torch.no_grad()
def lookahead_actions(agent, h, n, call_counter, samples, chunk=65536):
    """One-ply value look-ahead for the ``n`` envs of handle ``h``: int32 [n] actions maximising the mean
    over an action's expansion items of  q = reward + gamma * (1 - terminated) * V(successor)  (lowest
    action index on ties; action 0 for an env without a legal move).  Also returns the expansion and the
    per-(env, action) table q [n, 192] (-inf where an action is not legal)."""
    ex = h.expand(call_counter, samples)
    dev = ex["offsets"].device
    items = ex["action"].numel()
    q = torch.full((n * 192,), float("-inf"), dtype=torch.float32, device=dev)
    if items:
        v = agent.values({"board": ex["board"], "pieces": ex["pieces"], "mask": ex["mask"]}, chunk=chunk).reshape(-1)
        q_item = ex["reward"] + float(agent.config.gamma) * (1.0 - ex["terminated"].float()) * v.float()
        env = torch.repeat_interleave(torch.arange(n, device=dev), ex["offsets"].diff(), output_size=items)
        key = env * 192 + ex["action"].long()
        sums = torch.zeros(n * 192, dtype=torch.float32, device=dev).index_add_(0, key, q_item)
        cnt = torch.zeros(n * 192, dtype=torch.float32, device=dev).index_add_(0, key, torch.ones_like(q_item))
        q = torch.where(cnt > 0, sums / cnt.clamp(min=1.0), q)
    q = q.view(n, 192)
    return q.argmax(dim=1).to(torch.int32), ex, q


@torch.no_grad()
def evaluate(agent, num_episodes=100, seed=0, deterministic=True, max_steps=10000, reward_config=None,
             return_actions=False, lookahead=0):
    """``lookahead``: 0 = the agent's own policy (argmax when ``deterministic``); K >= 1 = one-ply value
    look-ahead with K sampled trios per dealing move (``lookahead_actions``, expansion call counter = the
    step number).  ``return_actions``: also return ``actions`` int32 [steps, n] (the action every env was given at every
    step; entries after an env's game over are ignored by the env) and ``rewards_per_episode`` — enough to
    replay every episode through another implementation of the rules (tests do, through the oracle)."""
    dev = agent.device
    n = int(num_episodes)
    h = capi.EnvHandle(n, seed, 0, reward_config, capi.ENV_NO_AUTO_RESET)
    board = torch.zeros(n, dtype=torch.int64, device=dev)
    pieces = torch.zeros(n, dtype=torch.int32, device=dev)
    mask = torch.zeros((3, n), dtype=torch.int64, device=dev)
    rewards = torch.zeros(n, dtype=torch.float32, device=dev)
    term = torch.zeros(n, dtype=torch.uint8, device=dev)
    total_reward = torch.zeros(n, dtype=torch.float64, device=dev)
    done = torch.zeros(n, dtype=torch.bool, device=dev)
    was_training = agent.training
    agent.eval()                                       # scripts/evaluate.py evaluates in eval mode
    steps = 0
    log = []
    while steps < max_steps and not bool(done.all()):
        if lookahead:
            act, _, _ = lookahead_actions(agent, h, n, steps, int(lookahead))
        else:
            h.observe(board, pieces, mask)
            act, _, _ = agent.act({"board": board, "pieces": pieces, "mask": mask}, deterministic=deterministic)
        if return_actions:
            log.append(act.clone())
        h.step(act, rewards, term, None, None, None, None)
        total_reward += torch.where(done, torch.zeros_like(rewards), rewards).double()
        done |= term.bool()
        steps += 1
    st = h.get_state()
    h.close()
    if was_training:
        agent.train()
    scores, lengths = st["score"].astype(np.int64), st["moves"].astype(np.int64)
    extra = {}
    if return_actions:
        extra = {"actions": torch.stack(log).cpu().numpy() if log else np.zeros((0, n), np.int32),
                 "rewards_per_episode": total_reward.cpu().numpy(), "lines": st["lines_total"].astype(np.int64),
                 "max_combos": st["max_streak"].astype(np.int64)}
    return {**extra, "num_episodes": n, "mean_score": float(scores.mean()), "std_score": float(scores.std()),
            "max_score": int(scores.max()), "min_score": int(scores.min()), "mean_length": float(lengths.mean()),
            "max_length": int(lengths.max()), "mean_lines": float(st["lines_total"].mean()),
            "max_combo": int(st["max_streak"].max()), "mean_reward": float(total_reward.mean().item()),
            "finished": int(done.sum().item()), "scores": scores, "lengths": lengths}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--checkpoint", required=True)
    ap.add_argument("--episodes", type=int, default=100)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--stochastic", action="store_true")
    ap.add_argument("--lookahead", type=int, default=0,
                    help="K >= 1: one-ply value look-ahead with K sampled trios per dealing move (0 = policy argmax)")
    a = ap.parse_args()
    agent = PPOAgent()
    agent.load(a.checkpoint)
    res = evaluate(agent, a.episodes, a.seed, deterministic=not a.stochastic, lookahead=a.lookahead)
    print(json.dumps({k: v for k, v in res.items() if not isinstance(v, np.ndarray)}, indent=1))


if __name__ == "__main__":
    main()
