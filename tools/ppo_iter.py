import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from bbgpu.ppo import PPOAgent, PPOConfig
from bbgpu.rollout import RolloutBuffer
from bbgpu.train import RolloutRunner
from bbgpu.vec_env import VectorizedBlockBlastEnv
dev = torch.device("cuda")
n, T, mb = 131072, 8, 32768
for fused_bn in (True, False):
    agent = PPOAgent(PPOConfig(batch_size=mb, num_epochs=2, precision="bf16", fused_bn=fused_bn), dev); agent.train()
    venv = VectorizedBlockBlastEnv(n, seed=1, output="packed")
    buf = RolloutBuffer(T, n, device=dev)
    runner = RolloutRunner(venv, agent, buf, use_graph=False)
    for it in range(4):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        last = runner.run()
        torch.cuda.synchronize(); t1 = time.perf_counter()
        m = agent.update(buf, last)
        torch.cuda.synchronize(); t2 = time.perf_counter()
        print("fused_bn=%s it %d collect %.3f s update %.3f s -> %.0f samples/s" % (fused_bn, it, t1 - t0, t2 - t1, n * T / (t2 - t0)), flush=True)
    venv.close(); del agent, buf
