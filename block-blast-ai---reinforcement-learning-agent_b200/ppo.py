"""PPO agent with action masking — the reference's ``PPOConfig`` / ``PPOAgent`` interface
(src/agents/ppo.py:26-449) on the device-resident path.

Collect: packed obs -> K2 (planes) -> CNN (PyTorch) -> K3 (masked sample + log-prob) -> K1
(env step), nothing leaves HBM.  Update: K4 GAE, whole-buffer advantage normalisation,
clipped surrogate + 0.5*MSE value loss + 0.01*entropy (ppo.py:372-392), grad-norm clip 0.5,
Adam(eps=1e-5).  With torch.distributed initialised every optimiser step all-reduces the
gradients in one flat NCCL bucket (dist.py); BatchNorm statistics stay per GPU (the
single-device reference has nothing to synchronise them with).
"""
from dataclasses import dataclass, field, fields
from typing import Tuple

import numpy as np
import torch

from . import capi, dist
from .network import BlockBlastNetwork, PPOLossTail, _pack_mask_planes
from .rollout import RolloutBuffer  # noqa: F401  (re-export, as in the reference module)


@dataclass
class PPOConfig:
    """Field names and defaults of the reference (ppo.py:26-46); ``precision`` is ours."""
    learning_rate: float = 3e-4
    gamma: float = 0.99
    gae_lambda: float = 0.95
    clip_epsilon: float = 0.2
    entropy_coef: float = 0.01
    value_coef: float = 0.5
    max_grad_norm: float = 0.5
    num_epochs: int = 10
    batch_size: int = 64
    conv_channels: Tuple[int, ...] = (64, 128, 128)
    fc_hidden: Tuple[int, ...] = (512, 256)
    precision: str = "fp32"          # "fp32" (reference numerics) | "bf16" (autocast, channels_last)
    fused_bn: bool = True            # bf16 only: BatchNorm + ReLU (+ residual add) as bb_bn_relu_* kernels around cuDNN's convs

    def to_dict(self):
        return {f.name: getattr(self, f.name) for f in fields(self)}

    @classmethod
    def from_dict(cls, data):
        names = {f.name for f in fields(cls)}
        return cls(**{k: v for k, v in data.items() if k in names})


class PPOAgent:
    def __init__(self, config=None, device=None, seed=0, global_env_offset=0):
        """``seed`` keys the action-sampling noise (with the global env id and a call counter, so
        that env shards on several GPUs draw independent noise and an N-GPU run samples what the
        1-GPU run samples); ``global_env_offset`` = global id of this rank's env 0."""
        if device is None:
            if not torch.cuda.is_available():
                raise capi.BBGpuError("PPOAgent needs a CUDA device (no CPU fallback)")
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = torch.device(device)
        self.config = config or PPOConfig()
        self.training = True
        self.network = BlockBlastNetwork(conv_channels=tuple(self.config.conv_channels),
                                         fc_hidden=tuple(self.config.fc_hidden)).to(self.device)
        if self.config.precision == "bf16":
            self.network = self.network.to(memory_format=torch.channels_last)
            self.network.set_fused_bn(self.config.fused_bn)
            torch.backends.cudnn.benchmark = True     # fixed shapes: let cuDNN pick the conv algorithms
        self.network.sample_seed = int(seed)
        self.network.sample_row_offset = int(global_env_offset)
        dist.broadcast_module(self.network)
        # fused=True: one multi-tensor kernel per step instead of a foreach sequence (same update rule)
        # capturable: the step counters live on the device, so the step can sit inside a CUDA graph
        self.optimizer = torch.optim.Adam(self.network.parameters(), lr=self.config.learning_rate, eps=1e-5,
                                          fused=self.device.type == "cuda", capturable=self.device.type == "cuda")
        self._graph = None
        self.scheduler = None
        # gradients of the FC encoder + heads (everything after the convolution stack in parameter order) are
        # reduced while backward is still in the convolutions
        n_conv = len(list(self.network.conv_encoder.parameters()))
        self.bucket = dist.FlatGradBucket(self.network.parameters(), early_from=n_conv)

    # ------------------------------------------------------------------ helpers
    def _autocast(self):
        return torch.autocast("cuda", dtype=torch.bfloat16, enabled=self.config.precision == "bf16")

    def _trunk(self, x):
        if self.config.precision == "bf16":
            x = x.contiguous(memory_format=torch.channels_last)
        with self._autocast():
            logits, value = self.network.trunk(x)
        return logits, value.float()

    def _obs_to_nchw(self, obs):
        """obs dict -> ((B,4,8,8) f32, mask planes int64 [3,B]) on the device.  Accepts the packed
        protocol ('board' int64[N], 'pieces' int32[N], 'mask' int64[3,N]) or dense arrays."""
        dev = self.device
        if "mask" in obs and isinstance(obs["board"], torch.Tensor) and obs["board"].dtype == torch.int64:
            n = obs["board"].shape[0]
            x = torch.empty((n, 4, 8, 8), dtype=torch.float32, device=dev)
            capi.unpack_obs(obs["board"], obs["pieces"], obs["mask"], obs["mask"].stride(0), obs=x, n=n)
            return x, obs["mask"]
        if "nchw" in obs:
            x = obs["nchw"]
        else:
            b = torch.as_tensor(np.asarray(obs["board"]) if not isinstance(obs["board"], torch.Tensor) else obs["board"]).to(dev).float()
            p = torch.as_tensor(np.asarray(obs["pieces"]) if not isinstance(obs["pieces"], torch.Tensor) else obs["pieces"]).to(dev).float()
            x = torch.cat([b.unsqueeze(1), p], dim=1)
        planes = None
        if "action_mask" in obs:
            m = obs["action_mask"]
            m = m if isinstance(m, torch.Tensor) else torch.as_tensor(np.asarray(m))
            planes = _pack_mask_planes(m.to(dev))
        return x, planes

    # ------------------------------------------------------------------ acting
    @torch.no_grad()
    def act(self, obs, deterministic=False, chunk=None):
        """Device fast path: returns (actions int32, log_probs, values) as CUDA tensors.
        ``chunk`` bounds the CNN batch (activation memory) for very large env counts; BatchNorm
        in train mode then uses per-chunk statistics."""
        x, planes = self._obs_to_nchw(obs)
        n = x.shape[0]
        if chunk is None or n <= chunk:
            logits, value = self._trunk(x)
        else:
            ls, vs = [], []
            for s0 in range(0, n, chunk):
                l, v = self._trunk(x[s0:s0 + chunk])
                ls.append(l)
                vs.append(v)
            logits, value = torch.cat(ls), torch.cat(vs)
        act, logp, _ = self.network.head_from_logits(logits, planes, None, deterministic, need_entropy=False)
        return act, logp, value

    @torch.no_grad()
    def act_into(self, obs, actions, log_probs, values, x_buf=None):
        """``act`` on a packed observation with caller-owned outputs (rows of a RolloutBuffer):
        K2 -> CNN -> K3 writing ``actions`` int32[N] / ``log_probs`` f32[N] in place, ``values`` f32[N]
        copied.  No allocation of result tensors, no host work besides the launches — the body of a
        captured rollout graph."""
        n = obs["board"].shape[0]
        x = x_buf if x_buf is not None else torch.empty((n, 4, 8, 8), dtype=torch.float32, device=self.device)
        capi.unpack_obs(obs["board"], obs["pieces"], obs["mask"], obs["mask"].stride(0), obs=x, n=n)
        logits, value = self._trunk(x)
        if logits.dtype not in (torch.float32, torch.bfloat16):
            logits = logits.float()
        net = self.network
        ctr = net.sample_counter(self.device)
        capi.masked_sample(logits.contiguous(), obs["mask"], obs["mask"].stride(0), net.sample_seed, 1, 0, actions,
                           log_probs, None, net.sample_row_offset, ctr)
        ctr.add_(1)
        values.copy_(value)

    def select_actions(self, observations, deterministic=False):
        """ppo.py:291-319: numpy in, numpy out."""
        act, logp, value = self.act(observations, deterministic)
        return act.cpu().numpy().astype(np.int64), logp.cpu().numpy(), value.cpu().numpy()

    def select_action(self, observation, deterministic=False):
        """ppo.py:261-289 (single observation)."""
        obs = {k: (v.unsqueeze(0) if isinstance(v, torch.Tensor) else np.asarray(v)[None]) for k, v in observation.items()
               if k in ("board", "pieces", "action_mask")}
        x, planes = self._obs_to_nchw(obs)
        with torch.no_grad():
            logits, value = self._trunk(x)
            act, logp, ent = self.network.head_from_logits(logits, planes, None, deterministic)
        return int(act.item()), {"log_prob": float(logp.item()), "entropy": float(ent.item()), "value": float(value.item())}

    @torch.no_grad()
    def values(self, obs, chunk=None):
        x, _ = self._obs_to_nchw({k: v for k, v in obs.items() if k != "action_mask"})
        if chunk is None or x.shape[0] <= chunk:
            return self._trunk(x)[1]
        return torch.cat([self._trunk(x[s0:s0 + chunk])[1] for s0 in range(0, x.shape[0], chunk)])

    def get_values(self, observations):
        """ppo.py:321-328."""
        return self.values(observations).cpu().numpy()

    # ------------------------------------------------------------------ update
    def _fused_step(self, obs, mask, actions, old_logp, adv, ret, sums):
        """One optimiser step on a gathered minibatch (fused loss tail); metric terms added to ``sums``."""
        cfg = self.config
        if cfg.precision == "bf16":
            obs = obs.contiguous(memory_format=torch.channels_last)
        with self._autocast():
            logits, values = self.network.trunk(obs)
        loss, means = PPOLossTail.apply(logits, values.float(), mask, actions, old_logp, adv, ret,
                                        cfg.clip_epsilon, cfg.value_coef, cfg.entropy_coef)
        self.bucket.zero()
        loss.backward()
        self.bucket.all_reduce_mean()                  # C1: one flat NCCL all-reduce
        self.bucket.clip_grad_norm_(cfg.max_grad_norm)
        self.optimizer.step()
        sums += torch.stack([means[0], means[1], means[2], loss.detach().double(), means[3], means[4]])

    def _minibatch(self, buffer, idx, mean_std, out, sums):
        """gather (bb_gather_minibatch) of samples ``idx``, then one optimiser step on them."""
        g = buffer.gather(idx, mean_std, out=out)
        self._fused_step(g["obs"], g["mask"], g["actions"], g["logp"], g["adv"], g["ret"], sums)

    def _graph_step(self, buffer):
        """The minibatch step as a replayable CUDA graph: gather (bb_gather_minibatch) of the static
        index tensor, CNN forward / backward, loss tail, gradient all-reduce, clip, Adam — ~250
        launches collapse into one graph launch, which is what bounds the reference's own schedule
        (2,048-sample minibatches) on a B200.  Captured once per (buffer, batch size)."""
        key = (id(buffer), self.config.batch_size)
        if self._graph is not None and self._graph["key"] == key:
            return self._graph
        dev, b = self.device, self.config.batch_size
        st = {"key": key, "idx": torch.zeros(b, dtype=torch.int64, device=dev),
              "ms": torch.zeros(2, dtype=torch.float32, device=dev),
              "sums": torch.zeros(6, dtype=torch.float64, device=dev)}
        st["out"] = buffer.gather(st["idx"], st["ms"])
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self._minibatch(buffer, st["idx"], st["ms"], st["out"], st["sums"])
        st["graph"] = graph
        self._graph = st
        return st

    def update(self, buffer, last_values, use_graph=False):
        """ppo.py:330-423.  Returns the reference's metric dict.  Every minibatch is ``_minibatch``;
        with ``use_graph`` and full minibatches it is replayed as a captured CUDA graph (the first
        update always runs eagerly so that cuDNN autotuning and the optimiser state exist before the
        capture)."""
        cfg = self.config
        buffer.compute_returns_and_advantages(last_values, cfg.gamma, cfg.gae_lambda)
        self.bucket.rebind()
        total, b = buffer.buffer_size * buffer.num_envs, cfg.batch_size
        self._updates_done = getattr(self, "_updates_done", 0) + 1
        graph = use_graph and total % b == 0 and self._updates_done > 1
        st = self._graph_step(buffer) if graph else None
        mean, std = buffer.advantage_mean_std()
        ms = torch.stack([mean, std]).float()
        if graph:
            st["ms"].copy_(ms)
            sums = st["sums"].zero_()
        else:
            sums = torch.zeros(6, dtype=torch.float64, device=self.device)
        n_updates = 0
        for _ in range(cfg.num_epochs):
            perm = torch.randperm(total, device=self.device)
            for start in range(0, total, b):
                if graph:
                    st["idx"].copy_(perm[start:start + b])
                    st["graph"].replay()
                else:
                    self._minibatch(buffer, perm[start:start + b], ms, None, sums)
                n_updates += 1
        s = (sums / max(n_updates, 1)).cpu().tolist()
        return {"policy_loss": s[0], "value_loss": s[1], "entropy": s[2], "total_loss": s[3],
                "approx_kl": s[4], "clip_fraction": s[5]}

    # ------------------------------------------------------------------ persistence / modes
    def save(self, path, network_state=None):
        """``network_state``: write this state_dict instead of the network's current one (best.pt snapshots).
        Same keys as ppo.py:425-431 so the reference's PPOAgent.load / evaluate.py / GUI can read
        it (tensors and plain Python values only: loads with torch.load(weights_only=True), the
        default of the reference's torch.load call).  The optimizer state is written in the form a
        plain torch.optim.Adam on any device accepts: CPU scalar ``step`` counters, no
        fused / foreach / capturable flags of ours.  ``b200_state`` (ignored by the reference)
        carries the sampling-noise position for --resume."""
        cfgd = {k: (list(v) if isinstance(v, tuple) else v) for k, v in self.config.to_dict().items()
                if k not in ("precision", "fused_bn")}
        opt = self.optimizer.state_dict()
        opt = {"state": {k: {n: (v.detach().cpu().float().reshape(()) if n == "step" and torch.is_tensor(v) else v)
                             for n, v in st.items()} for k, st in opt["state"].items()},
               "param_groups": [{**g, "fused": None, "foreach": None, "capturable": False} for g in opt["param_groups"]]}
        torch.save({"network_state_dict": network_state if network_state is not None else self.network.state_dict(),
                    "optimizer_state_dict": opt, "config": cfgd,
                    "b200_state": {"sample_calls": self.network.sample_calls, "sample_seed": self.network.sample_seed}},
                   path)

    def load(self, path):
        ck = torch.load(path, map_location=self.device, weights_only=True)
        self.network.load_state_dict(ck["network_state_dict"])
        if "optimizer_state_dict" in ck:
            opt = ck["optimizer_state_dict"]
            mine = self.optimizer.state_dict()["param_groups"]
            # keep this optimizer's own execution flags (fused / capturable), take the hyper-parameters
            groups = [{**g, **{k: m[k] for k in ("fused", "foreach", "capturable") if k in m}}
                      for g, m in zip(opt["param_groups"], mine)]
            self.optimizer.load_state_dict({"state": opt["state"], "param_groups": groups})
        if "config" in ck:
            cfg = {k: (tuple(v) if isinstance(v, list) else v) for k, v in ck["config"].items()}
            self.config = PPOConfig.from_dict({**cfg, "precision": self.config.precision,
                                               "fused_bn": self.config.fused_bn})
        if "b200_state" in ck:
            self.network.sample_calls = ck["b200_state"].get("sample_calls", 0)
        self.bucket.rebind()
        self._graph = None          # a captured minibatch step has the old hyper-parameters baked in

    def train(self):
        self.training = True
        self.network.train()

    def eval(self):
        self.training = False
        self.network.eval()
