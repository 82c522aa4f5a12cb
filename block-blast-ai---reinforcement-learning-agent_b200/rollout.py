"""Device-resident rollout buffer with the reference's ``RolloutBuffer`` interface
(src/agents/ppo.py:70-218).

Storage is the packed protocol — per sample: board u64, pieces u32, mask 3 x u64, action i32
and five f32 scalars (reward, done, value, log-prob; advantage/return computed later) = 64 B
instead of the reference's 1,824 B of float planes, so 131,072 envs x 128 steps is 1.07 GB
and never leaves HBM.  ``compute_returns_and_advantages`` is the K4 kernel (bit-identical to
ppo.py:141-169); ``get_samples`` yields the reference's 7-tuple with the float planes
expanded on the fly by K2; the whole-buffer advantage normalisation (ppo.py:196) uses K4's
float64 moments, all-reduced across ranks when torch.distributed is initialised.
"""
import numpy as np
import torch

from . import capi


def _to_dev(x, device, dtype):
    if isinstance(x, torch.Tensor):
        return x.to(device=device, dtype=dtype, non_blocking=True)
    return torch.as_tensor(np.asarray(x), device=device).to(dtype)


def pack_dense_obs(board, pieces_planes, action_mask, device):
    """Reference-layout observation (board (N,8,8), pieces (N,3,8,8), action_mask (N,192)) ->
    the packed protocol the env writes: board int64[N], pieces word int32[N] (piece ids in bytes
    0-2, used flags in bits 24-26), mask planes int64[3,N].  Each piece plane is looked up in the
    library's piece table; an all-zero plane is a used slot.  Raises ValueError for a plane that
    is not one of the 37 pieces drawn at the origin."""
    w = (2 ** torch.arange(64, device=device, dtype=torch.int64))          # bit weights (wraps at 2**63)
    b = (_to_dev(board, device, torch.float32).reshape(-1, 64) != 0).to(torch.int64)
    p = (_to_dev(pieces_planes, device, torch.float32).reshape(-1, 3, 64) != 0).to(torch.int64)
    m = (_to_dev(action_mask, device, torch.float32).reshape(-1, 3, 64) != 0).to(torch.int64)
    planes = (p * w).sum(-1)                                                # [N,3]
    table = torch.as_tensor(capi.piece_table()[0].view(np.int64), device=device)
    hit = planes.unsqueeze(-1) == table                                     # [N,3,37]; the 37 masks are distinct
    used = planes == 0
    if bool((~used & ~hit.any(-1)).any()):
        raise ValueError("RolloutBuffer.add: a piece plane is neither empty nor a piece at the origin")
    ids = (hit.to(torch.int64) * torch.arange(37, device=device)).sum(-1)   # 0 for a used slot
    k = torch.arange(3, device=device)
    word = ((ids << (8 * k)) | (used.to(torch.int64) << (24 + k))).sum(-1).to(torch.int32)
    return (b * w).sum(-1), word, (m * w).sum(-1).t().contiguous()


class RolloutBuffer:
    def __init__(self, buffer_size, num_envs, board_size=8, num_pieces=3, action_space_size=192,
                 device=None):
        assert board_size == 8 and num_pieces == 3 and action_space_size == 192
        if device is None or torch.device(device).type != "cuda":
            if not torch.cuda.is_available():
                raise capi.BBGpuError("RolloutBuffer lives in GPU memory; no CUDA device available")
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = torch.device(device)
        self.buffer_size, self.num_envs = int(buffer_size), int(num_envs)
        T, N, dev = self.buffer_size, self.num_envs, self.device
        # T+1 observation rows: row t is the observation the action of step t was chosen on, row T the
        # one after the last step.  On the device-resident path the step kernel writes row t+1 itself
        # (obs_row), so collecting a rollout copies nothing.
        self.boards = torch.zeros((T + 1, N), dtype=torch.int64, device=dev)
        self.pieces = torch.zeros((T + 1, N), dtype=torch.int32, device=dev)
        self.action_masks = torch.zeros((T + 1, 3, N), dtype=torch.int64, device=dev)
        self.terminated = torch.zeros((T, N), dtype=torch.uint8, device=dev)   # raw done flags of the step kernel
        self.actions = torch.zeros((T, N), dtype=torch.int32, device=dev)
        self.log_probs = torch.zeros((T, N), dtype=torch.float32, device=dev)
        self.rewards = torch.zeros((T, N), dtype=torch.float32, device=dev)
        self.dones = torch.zeros((T, N), dtype=torch.float32, device=dev)
        self.values = torch.zeros((T, N), dtype=torch.float32, device=dev)
        self.advantages = torch.zeros((T, N), dtype=torch.float32, device=dev)
        self.returns = torch.zeros((T, N), dtype=torch.float32, device=dev)
        self.moments = torch.zeros(2, dtype=torch.float64, device=dev)
        self.ptr, self.full = 0, False

    # ------------------------------------------------------------------ filling
    def add(self, board, pieces, action_mask, action, log_prob, reward, done, value):
        """ppo.py:116-139.  Accepts either packed tensors (board int64[N], pieces int32[N],
        action_mask int64[3,N]) or the reference's dense arrays, which are packed on the way in."""
        t, dev = self.ptr, self.device
        if not (isinstance(board, torch.Tensor) and board.dtype == torch.int64 and board.dim() == 1):
            board, pieces, action_mask = pack_dense_obs(board, pieces, action_mask, dev)
        self.boards[t].copy_(board, non_blocking=True)
        self.pieces[t].copy_(pieces, non_blocking=True)
        self.action_masks[t].copy_(action_mask, non_blocking=True)
        self.actions[t] = _to_dev(action, dev, torch.int32)
        self.log_probs[t] = _to_dev(log_prob, dev, torch.float32)
        self.rewards[t] = _to_dev(reward, dev, torch.float32)
        self.dones[t] = _to_dev(done, dev, torch.float32)
        self.values[t] = _to_dev(value, dev, torch.float32)
        self.ptr += 1
        if self.ptr >= self.buffer_size:
            self.full = True

    def obs_row(self, t):
        """Packed observation row t (0..T) as the dict the env / agent exchange (views, no copies)."""
        return {"board": self.boards[t], "pieces": self.pieces[t], "mask": self.action_masks[t]}

    def set_first_obs(self, obs):
        if obs["board"].data_ptr() != self.boards[0].data_ptr():
            self.boards[0].copy_(obs["board"], non_blocking=True)
            self.pieces[0].copy_(obs["pieces"], non_blocking=True)
            self.action_masks[0].copy_(obs["mask"], non_blocking=True)

    def finish_direct(self):
        """After a rollout written in place (train.RolloutRunner): done flags u8 -> f32, buffer full."""
        self.dones.copy_(self.terminated)
        self.ptr, self.full = self.buffer_size, True

    def reset(self):
        self.ptr, self.full = 0, False

    # ------------------------------------------------------------------ GAE (K4)
    def compute_returns_and_advantages(self, last_values, gamma, gae_lambda):
        """ppo.py:141-169 on the device; also refreshes the advantage moments."""
        lv = _to_dev(last_values, self.device, torch.float32).contiguous()
        self.moments.zero_()
        capi.gae(self.rewards, self.values, self.dones, lv, gamma, gae_lambda, self.advantages, self.returns,
                 self.moments)

    def advantage_mean_std(self):
        """Whole-buffer mean and population std (ppo.py:196), over all ranks."""
        m = self.moments.clone()
        cnt = torch.tensor([float(self.buffer_size * self.num_envs)], dtype=torch.float64, device=self.device)
        if torch.distributed.is_available() and torch.distributed.is_initialized() and torch.distributed.get_world_size() > 1:
            pack = torch.cat([m, cnt])
            torch.distributed.all_reduce(pack)
            m, cnt = pack[:2], pack[2:]
        mean = m[0] / cnt[0]
        var = (m[1] / cnt[0] - mean * mean).clamp(min=0.0)
        return mean.float(), var.sqrt().float()

    # ------------------------------------------------------------------ minibatches
    def gather(self, idx, mean_std, obs_dtype=torch.float32, out=None):
        """Minibatch ``idx`` (int64 flat sample indices) of the packed buffer in ONE library call
        (bb_gather_minibatch): obs planes (B,4,8,8), mask planes int64 [3,B], actions int32, old
        log-probs, advantages normalised with ``mean_std`` (float32 [2] device tensor), returns.
        ``out``: a dict of preallocated outputs to fill (static buffers of a captured CUDA graph)."""
        b, dev = idx.numel(), self.device
        if out is None:
            out = dict(obs=torch.empty((b, 4, 8, 8), dtype=obs_dtype, device=dev),
                       mask=torch.empty((3, b), dtype=torch.int64, device=dev),
                       actions=torch.empty(b, dtype=torch.int32, device=dev),
                       logp=torch.empty(b, dtype=torch.float32, device=dev),
                       adv=torch.empty(b, dtype=torch.float32, device=dev),
                       ret=torch.empty(b, dtype=torch.float32, device=dev))
        capi.gather_minibatch(idx, self.num_envs, self.boards, self.pieces, self.action_masks, self.actions,
                              self.log_probs, self.advantages, self.returns, mean_std, out["obs"], out["mask"],
                              out["actions"], out["logp"], out["adv"], out["ret"])
        return out

    def get_samples(self, batch_size):
        """ppo.py:171-213: yields (boards (B,8,8), pieces (B,3,8,8), action_masks (B,192) f32,
        actions int64, old_log_probs, advantages, returns) in the reference's layouts (CUDA
        tensors), one ``gather`` per minibatch of a random permutation."""
        total = self.buffer_size * self.num_envs
        mean, std = self.advantage_mean_std()
        ms = torch.stack([mean, std])
        perm = torch.randperm(total, device=self.device)
        for start in range(0, total, batch_size):
            g = self.gather(perm[start:start + batch_size], ms)
            b = g["actions"].numel()
            dense = torch.empty((b, 192), dtype=torch.float32, device=self.device)
            capi.unpack_obs(None, None, g["mask"], b, mask_dense=dense, n=b)
            yield g["obs"][:, 0], g["obs"][:, 1:], dense, g["actions"].long(), g["logp"], g["adv"], g["ret"]
