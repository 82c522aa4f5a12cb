"""Masked-PPO training loop on the device-resident path — the reference's
``scripts/train.py:train`` (lines 60-316) with the same config keys, loop shape, metric names
and checkpoint files, run by one process per GPU.

    python -m bbgpu.train --config cfg.yaml [--resume ckpt.pt] [--seed 42]
    torchrun --nproc-per-node 8 -m bbgpu.train --config cfg.yaml        (config 4 / 5)

Config quirks of the reference are honoured (SURVEY.md §5): ``num_epochs`` is read from the
``ppo`` section (both shipped YAMLs put it under ``training``, so the default 10 applies),
``batch_size`` from ``training``, the ``network`` / ``environment`` sections are ignored.
Keys of ours live under ``b200:`` (precision, reseed_on_reset, log_every_update, symmetrize, canonical_frame).
"""
import argparse
import json
import os
import time

import numpy as np
import torch

from . import dist
from .logger import Logger, TensorBoardLogger, tensorboard_tags
from .ppo import PPOAgent, PPOConfig
from .rollout import RolloutBuffer
from .vec_env import VectorizedBlockBlastEnv


def load_config(path):
    import yaml
    with open(path) as f:
        return yaml.safe_load(f)


def set_seed(seed):
    np.random.seed(seed)
    torch.manual_seed(seed)
    torch.cuda.manual_seed_all(seed)


class RolloutRunner:
    """The collect phase of scripts/train.py:173-207 with every result written in place: K2 -> CNN ->
    K3 put action / log-prob / value straight into row t of the RolloutBuffer, K1 puts reward, done flag
    and the packed next observation into rows t / t+1, and the episode statistics the reference reads from
    ``infos`` (train.py:196-201) accumulate inside K1 (``vec_env.episode_stats``).  Nothing is copied and
    nothing leaves the device.  With ``use_graph`` the whole T-step rollout plus the bootstrap value pass
    is captured once as ONE CUDA graph and replayed — at the reference's 64 envs per process the step is
    ~60 launches of a few microseconds each, i.e. launch-bound when issued from Python."""

    def __init__(self, vec_env, agent, buffer, use_graph=True):
        self.vec_env, self.agent, self.buffer = vec_env, agent, buffer
        n, dev = buffer.num_envs, buffer.device
        rows = 8 * n if agent.config.symmetrize else n            # symmetrize: the eight views of every env
        self.x_buf = torch.empty((rows, 4, 8, 8), dtype=torch.float32, device=dev)
        # canonical_frame: static canonical rows and view sets of the n envs, so that the rollout graph captures them
        self.canon = ((torch.empty(n, dtype=torch.int64, device=dev), torch.empty(n, dtype=torch.int32, device=dev),
                       torch.empty(n, dtype=torch.uint8, device=dev)) if agent.config.canonical_frame else None)
        self.last_values = torch.zeros(n, dtype=torch.float32, device=dev)
        self.use_graph, self.graph, self.calls = bool(use_graph), None, 0

    def _body(self):
        buf, T = self.buffer, self.buffer.buffer_size
        buf.set_first_obs(buf.obs_row(T))                      # continue from the last observation
        for t in range(T):
            self.agent.act_into(buf.obs_row(t), buf.actions[t], buf.log_probs[t], buf.values[t], self.x_buf, self.canon)
            self.vec_env.step_into(buf.actions[t], buf.rewards[t], buf.terminated[t], buf.obs_row(t + 1))
        self.last_values.copy_(self.agent.values(buf.obs_row(T)))
        buf.finish_direct()

    def run(self):
        """One rollout; returns the bootstrap values of the observation after the last step."""
        buf = self.buffer
        if self.calls == 0:
            self.vec_env.current_obs_into(buf.obs_row(buf.buffer_size))
        self.calls += 1
        if self.use_graph and self.calls > 1:                  # first rollout eager: cuDNN autotuning, allocator
            if self.graph is None:
                self.graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.graph):
                    self._body()
            self.graph.replay()
            buf.ptr, buf.full = buf.buffer_size, True
        else:
            self._body()
        return self.last_values

    def episode_stats(self):
        """(episodes, sum of final scores, max final score, sum of lengths) since the last call."""
        st = self.vec_env.episode_stats
        v = st.tolist()
        st.zero_()
        return v[1], v[2], v[4], v[3]


def train(config, resume_path=None, seed=42, progress_callback=None, max_updates=None):
    rank, world, local = dist.init()
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    set_seed(seed + rank)
    ppo_c, tr_c = config.get("ppo", {}), config.get("training", {})
    rew_c, log_c, ours = config.get("rewards", {}), config.get("logging", {}), config.get("b200", {})
    paths = config.get("paths", {})
    ckpt_dir, log_dir = paths.get("checkpoint_dir", "checkpoints"), paths.get("log_dir", "logs")
    if rank == 0:
        os.makedirs(ckpt_dir, exist_ok=True)
        os.makedirs(log_dir, exist_ok=True)

    num_envs = tr_c.get("num_envs", 64)                       # whole job; sharded over ranks
    if num_envs % world:
        # unequal shards would give the ranks different minibatch counts, i.e. different numbers of
        # gradient all-reduces per epoch (a hang), and unequal weights in the gradient mean
        raise ValueError("training.num_envs (%d) must be divisible by the number of GPUs (%d)" % (num_envs, world))
    offset, n_local = dist.shard(num_envs)
    # b200.stream_period = P: env g draws its pieces from stream g mod P, i.e. the job plays num_envs / P copies of
    # the same P piece streams (with reseed_on_reset: the reference's 64 fixed games, several trajectories of each
    # per update); the action-sampling noise stays keyed by the true global env id, so the copies explore differently
    period = int(ours.get("stream_period", 0) or 0)
    if period and (period % n_local or num_envs % period):
        raise ValueError("b200.stream_period (%d) must be a multiple of the envs per GPU (%d) and divide num_envs" % (period, n_local))
    vec_env = VectorizedBlockBlastEnv(n_local, seed=seed, reward_config=rew_c or None, output="packed",
                                      global_env_offset=offset % period if period else offset,
                                      reseed_on_reset=bool(ours.get("reseed_on_reset", False)))
    agent = PPOAgent(PPOConfig(
        learning_rate=ppo_c.get("learning_rate", 3e-4), gamma=ppo_c.get("gamma", 0.99),
        gae_lambda=ppo_c.get("gae_lambda", 0.95), clip_epsilon=ppo_c.get("clip_epsilon", 0.2),
        entropy_coef=ppo_c.get("entropy_coef", 0.01), value_coef=ppo_c.get("value_coef", 0.5),
        max_grad_norm=ppo_c.get("max_grad_norm", 0.5), num_epochs=ppo_c.get("num_epochs", 10),
        batch_size=tr_c.get("batch_size", 2048), precision=ours.get("precision", "fp32"),
        symmetrize=bool(ours.get("symmetrize", False)), canonical_frame=bool(ours.get("canonical_frame", False))), device,
        seed=seed, global_env_offset=offset)                  # sampling noise keyed by (seed, GLOBAL env id, call)
    agent.train()                                             # train mode during rollout too (scripts/train.py:122)
    start_step = 0
    if resume_path and os.path.exists(resume_path):
        agent.load(resume_path)
        for k in ("symmetrize", "canonical_frame"):           # the config's policy form wins over the checkpoint's
            if k in ours:
                setattr(agent.config, k, bool(ours[k]))
        if agent.config.symmetrize and agent.config.canonical_frame:   # one from the checkpoint, one from the config
            setattr(agent.config, "canonical_frame" if "symmetrize" in ours else "symmetrize", False)
        try:
            start_step = int(os.path.splitext(os.path.basename(resume_path))[0].split("_")[-1])
        except ValueError:
            pass
    rollout_steps = tr_c.get("rollout_steps", 128)
    buffer = RolloutBuffer(rollout_steps, n_local, device=device)
    total_timesteps = tr_c.get("total_timesteps", 50_000_000)
    log_interval, save_interval = log_c.get("log_interval", 100), log_c.get("save_interval", 1000)

    vec_env.reset()
    use_graph = bool(ours.get("cuda_graph", True))
    graph_update = bool(ours.get("cuda_graph_update", use_graph))   # the minibatch step (with its NCCL all-reduce) as a graph
    runner = RolloutRunner(vec_env, agent, buffer, use_graph)
    target_score = ours.get("stop_at_avg_score")              # optional early stop (score-vs-wallclock runs)
    max_wall_s = ours.get("max_wall_s")                       # optional wall-clock budget
    best_every_s = float(ours.get("best_save_min_interval_s", 10.0))
    global_step, num_updates, best_score, recent = start_step, 0, 0.0, []
    best_state, best_saved_at = None, 0.0
    history = []
    # same files / keys / TensorBoard tags as scripts/train.py:136-137, 231-258 (rank 0 only)
    logger = Logger(log_dir, name="ppo_b200") if rank == 0 else None
    tb_logger = TensorBoardLogger(log_dir, name="ppo_b200") if rank == 0 and log_c.get("tensorboard", True) else None
    t0 = time.time()
    try:
        while global_step < total_timesteps:
            last_values = runner.run()
            global_step += num_envs * rollout_steps
            metrics = agent.update(buffer, last_values, use_graph=graph_update)
            num_updates += 1
            e_cnt, e_sum, e_max, e_len = runner.episode_stats()
            cnt, ssum, lsum = dist.all_reduce_scalars([e_cnt, e_sum, e_len], device=device)
            # the wall clock is reduced too: every rank must take the same stop decision (a rank that leaves the
            # loop one update early would leave the others waiting in the next gradient all-reduce)
            smax, elapsed = dist.all_reduce_scalars([e_max, time.time() - t0], op="max", device=device)
            avg_score = ssum / cnt if cnt else 0.0
            recent.append((cnt, ssum))
            del recent[:-10]
            avg10 = sum(x[1] for x in recent) / max(sum(x[0] for x in recent), 1)     # episodes of the last 10 updates
            row = {"step": global_step, "fps": (global_step - start_step) / max(elapsed, 1e-9), "avg_score": avg_score,
                   "max_score": smax, "best_score": max(best_score, avg_score), "avg_length": lsum / cnt if cnt else 0.0,
                   "episodes": cnt, "wall_s": elapsed, "avg_score_10_updates": avg10, **metrics}
            history.append(row)
            stop = bool((max_updates and num_updates >= max_updates) or (max_wall_s and elapsed >= max_wall_s) or
                        (target_score and len(recent) == 10 and avg10 >= target_score) or global_step >= total_timesteps)
            if rank == 0:
                if avg_score > best_score:
                    # snapshot the weights on the device now (cheap), write best.pt at most every few seconds:
                    # an update takes tens of milliseconds here and early on nearly every one is a new best
                    best_score = avg_score
                    best_state = {k: v.detach().clone() for k, v in agent.network.state_dict().items()}
                if best_state is not None and time.time() - best_saved_at > best_every_s:
                    agent.save(os.path.join(ckpt_dir, "best.pt"), network_state=best_state)
                    best_state, best_saved_at = None, time.time()
                if num_updates % log_interval == 0 or num_updates <= 10 or ours.get("log_every_update") or stop:
                    logger.log(row, global_step)
                    if tb_logger is not None:
                        tb_logger.log_metrics(tensorboard_tags(row), global_step)
                    print("update %d step=%d fps=%.0f avg_score=%.1f max=%d len=%.1f entropy=%.3f kl=%.4f clip=%.3f"
                          % (num_updates, global_step, row["fps"], avg_score, smax, row["avg_length"], metrics["entropy"],
                             metrics["approx_kl"], metrics["clip_fraction"]), flush=True)
                if num_updates % save_interval == 0:
                    agent.save(os.path.join(ckpt_dir, "checkpoint_%d.pt" % global_step))
                    agent.save(os.path.join(ckpt_dir, "latest.pt"))
            if progress_callback is not None and not progress_callback(
                    {"total_steps": global_step, "mean_score": avg_score, "best_score": best_score,
                     "episodes": cnt, "fps": row["fps"]}):
                break
            if max_updates and num_updates >= max_updates:
                break
            if target_score and len(recent) == 10 and avg10 >= target_score:
                break
            if max_wall_s and elapsed >= max_wall_s:
                break
    finally:
        if rank == 0:
            if best_state is not None:
                agent.save(os.path.join(ckpt_dir, "best.pt"), network_state=best_state)
            agent.save(os.path.join(ckpt_dir, "final.pt"))
            if logger.metrics_history:
                logger.save_summary()
            if tb_logger is not None:
                tb_logger.close()
        vec_env.close()
    return history


def main():
    ap = argparse.ArgumentParser(description="B200 masked-PPO training for Block Blast")
    ap.add_argument("--config", required=True)
    ap.add_argument("--resume", default=None)
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--max-updates", type=int, default=None)
    a = ap.parse_args()
    train(load_config(a.config), a.resume, a.seed, max_updates=a.max_updates)
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
