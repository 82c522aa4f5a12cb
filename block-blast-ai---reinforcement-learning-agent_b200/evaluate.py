"""Batched evaluation of a trained agent — the reference's ``scripts/evaluate.py:23-90``
(one env, ``deterministic=True`` argmax rollouts) run for many episodes at once on the GPU.

Each of ``num_episodes`` envs plays exactly one episode (``BB_ENV_NO_AUTO_RESET``: a finished env
stays GAME_OVER and its further steps are no-ops), so the returned statistics are per-episode
like the reference's: scores, lengths, lines cleared, max combo.  The argmax policy runs the network only
on the episodes that are still going (``bb_env_observe_live`` compacts their observations each step).

    python -m bbgpu.evaluate --checkpoint checkpoints/best.pt --episodes 1000

``--lookahead K`` (K >= 1) replaces the argmax policy by a one-ply value look-ahead: every legal move
of every env is expanded on the GPU (``bb_env_expand``; a move that places the last piece is dealt K
sampled trios from the look-ahead stream, never the env's own), the successors are scored by the value
head, and each env plays the move with the highest mean ``reward + gamma * (1 - terminated) * V``.

``--symmetrize`` evaluates the agent's policy and value as averages over the eight board symmetries
(``PPOConfig.symmetrize``) even when the checkpoint was trained without them; ``--canonical-frame`` evaluates
them on the canonical view of each state instead (``PPOConfig.canonical_frame``, one network row per state).
By default the checkpoint's own setting applies.
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


def live_rows(m, n):
    """Network rows for ``m`` live envs of ``n``: ``m`` rounded up to one of four sizes per octave (at most n).
    It bounds the number of distinct batch shapes cuDNN plans for (and, with ``cudnn.benchmark``, times) to
    about four per octave, at most a quarter more rows than ``m``."""
    q = 1 << max(m.bit_length() - 3, 0)
    return min(n, -(-m // q) * q)


@torch.no_grad()
def evaluate(agent, num_episodes=100, seed=0, deterministic=True, max_steps=10000, reward_config=None,
             return_actions=False, lookahead=0, symmetrize=None, canonical_frame=None, global_env_offset=0):
    """``lookahead``: 0 = the agent's own policy (argmax when ``deterministic``); K >= 1 = one-ply value
    look-ahead with K sampled trios per dealing move (``lookahead_actions``, expansion call counter = the
    step number).  ``return_actions``: also return ``actions`` int32 [steps, n] (the action every env was given at every
    step; entries after an env's game over are ignored by the env) and ``rewards_per_episode`` — enough to
    replay every episode through another implementation of the rules (tests do, through the oracle).
    ``symmetrize``: None = the agent's own setting; True / False = with / without the eight-view average for
    this evaluation (the successor values of ``lookahead`` included).  ``canonical_frame``: the same for the
    canonical-frame policy.  Turning one of the two on turns the other off for this evaluation; the agent's
    own settings are restored afterwards.  ``global_env_offset``: global id of episode 0, so that each rank's shard
    plays the games that episodes ``global_env_offset ...`` of one single-process evaluation would play.

    The deterministic policy (``lookahead`` 0) runs the network on the unfinished episodes only
    (``bb_env_observe_live``); the other paths run it on every episode at every step."""
    if symmetrize and canonical_frame:
        raise ValueError("evaluate: symmetrize and canonical_frame are mutually exclusive")
    dev = agent.device
    n = int(num_episodes)
    h = capi.EnvHandle(n, seed, global_env_offset, reward_config, capi.ENV_NO_AUTO_RESET)
    board = torch.zeros(n, dtype=torch.int64, device=dev)
    pieces = torch.zeros(n, dtype=torch.int32, device=dev)
    mask = torch.zeros((3, n), dtype=torch.int64, device=dev)
    rewards = torch.zeros(n, dtype=torch.float32, device=dev)
    term = torch.zeros(n, dtype=torch.uint8, device=dev)
    total_reward = torch.zeros(n, dtype=torch.float64, device=dev)
    done = torch.zeros(n, dtype=torch.bool, device=dev)
    was_training, was_sym, was_canon = agent.training, agent.config.symmetrize, agent.config.canonical_frame
    if symmetrize is not None:
        agent.config.symmetrize = bool(symmetrize)
        if symmetrize:
            agent.config.canonical_frame = False
    if canonical_frame is not None:
        agent.config.canonical_frame = bool(canonical_frame)
        if canonical_frame:
            agent.config.symmetrize = False
    agent.eval()                                       # scripts/evaluate.py evaluates in eval mode
    steps = 0
    log = []
    # K3 keys its sampling noise by row index: compacting the rows would change which draws a seeded
    # stochastic evaluation makes, so only the deterministic policy runs on the live rows
    compact = deterministic and not lookahead
    if compact:
        ids = torch.zeros(n, dtype=torch.int32, device=dev)
        count = torch.zeros(1, dtype=torch.int32, device=dev)
        act = torch.zeros(n, dtype=torch.int32, device=dev)
    try:
        while steps < max_steps:
            if compact:
                # the live rows, then one 4-byte read: the host synchronisation of the step
                h.observe_live(board, pieces, mask, ids, count)
                m = int(count.item())
                if m == 0:
                    break
                rows = live_rows(m, n)          # rows m..rows-1 hold observations of earlier steps; dropped below
                a, _, _ = agent.act({"board": board[:rows], "pieces": pieces[:rows], "mask": mask[:, :rows]},
                                    deterministic=True)
                # a finished env keeps its last action, which BB_ENV_NO_AUTO_RESET ignores
                act.index_copy_(0, ids[:m].long(), a[:m])
            else:
                if bool(done.all()):
                    break
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
    finally:
        # the caller's agent keeps its own policy form and mode whatever happens during the evaluation
        h.close()
        agent.config.symmetrize, agent.config.canonical_frame = was_sym, was_canon
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
    ap.add_argument("--symmetrize", action="store_true", default=None,
                    help="average the policy / value over the 8 board symmetries (default: the checkpoint's setting)")
    ap.add_argument("--canonical-frame", action="store_true", default=None,
                    help="evaluate the network on the canonical view of each state, mapped back (default: the "
                         "checkpoint's setting)")
    a = ap.parse_args()
    agent = PPOAgent()
    agent.load(a.checkpoint)
    res = evaluate(agent, a.episodes, a.seed, deterministic=not a.stochastic, lookahead=a.lookahead,
                   symmetrize=a.symmetrize, canonical_frame=a.canonical_frame)
    print(json.dumps({k: v for k, v in res.items() if not isinstance(v, np.ndarray)}, indent=1))


if __name__ == "__main__":
    main()
