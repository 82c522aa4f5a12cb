#!/usr/bin/env python3
"""Where does a PPO minibatch step spend its time? (GPU box)"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from bbgpu.network import PPOLossTail
from bbgpu.ppo import PPOAgent, PPOConfig
from bbgpu.rollout import RolloutBuffer
from bbgpu.train import RolloutRunner
from bbgpu.vec_env import VectorizedBlockBlastEnv
bench = "--bench" in sys.argv
torch.backends.cudnn.benchmark = bench
dev = torch.device("cuda")
n, T, mb = 65536, 8, 32768
agent = PPOAgent(PPOConfig(batch_size=mb, num_epochs=1, precision="bf16"), dev); agent.train()
cfg = agent.config
venv = VectorizedBlockBlastEnv(n, seed=1, output="packed")
buf = RolloutBuffer(T, n, device=dev)
runner = RolloutRunner(venv, agent, buf, use_graph=False)
for it in range(2):
    torch.cuda.synchronize(); t0 = time.perf_counter()
    last = runner.run()
    torch.cuda.synchronize(); t1 = time.perf_counter()
    m = agent.update(buf, last)
    torch.cuda.synchronize(); t2 = time.perf_counter()
print("cudnn.benchmark=%s collect %.3f s  update %.3f s (%d minibatches of %d -> %.1f ms each)" % (bench, t1 - t0, t2 - t1, n * T // mb, mb, (t2 - t1) / (n * T // mb) * 1e3))


def trunk_forward(g):
    o = g["obs"].contiguous(memory_format=torch.channels_last)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        logits, v = agent.network.trunk(o)
    return logits, v


def loss_tail(g, logits, v):
    return PPOLossTail.apply(logits, v.float(), g["mask"], g["actions"], g["logp"], g["adv"], g["ret"],
                             cfg.clip_epsilon, cfg.value_coef, cfg.entropy_coef)[0]


# breakdown of one minibatch
mean, std = buf.advantage_mean_std()
ms = torch.stack([mean, std]).float()
idx = torch.randperm(n * T, device=dev)[:mb]
torch.cuda.synchronize(); t0 = time.perf_counter()
g = buf.gather(idx, ms)
torch.cuda.synchronize(); t1 = time.perf_counter()
logits, v = trunk_forward(g)
torch.cuda.synchronize(); t2 = time.perf_counter()
agent.bucket.zero()
loss_tail(g, logits, v).backward()
torch.cuda.synchronize(); t3 = time.perf_counter()
agent.bucket.clip_grad_norm_(cfg.max_grad_norm); agent.optimizer.step()
torch.cuda.synchronize(); t4 = time.perf_counter()
print("minibatch: gather %.1f ms | trunk forward %.1f ms | PPOLossTail + backward %.1f ms | clip+adam %.1f ms" % ((t1 - t0) * 1e3, (t2 - t1) * 1e3, (t3 - t2) * 1e3, (t4 - t3) * 1e3))
from torch.profiler import profile, ProfilerActivity
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    logits, v = trunk_forward(g)
    loss_tail(g, logits, v).backward()
    torch.cuda.synchronize()
print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=14, max_name_column_width=70))
