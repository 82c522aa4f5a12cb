"""ctypes binding of libbbgpu.so (C ABI: include/bbgpu.h).

Loads the in-tree CUDA library and fails loudly when it is missing — there is no CPU
fallback anywhere in this package.  PyTorch is used only for device memory and streams:
every ``torch.Tensor`` argument is passed as ``tensor.data_ptr()``.
"""
import ctypes as C
import os

import numpy as np

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BBGPU_LIB") or os.path.join(PKG_DIR, "libbbgpu.so")   # BBGPU_LIB: tuning builds only

BB_F32, BB_BF16, BB_U8 = 0, 1, 2
ENV_RESEED_ON_RESET = 1
ENV_NO_AUTO_RESET = 2
ABI_VERSION = 2

REWARD_KEYS = ("line_clear_base", "block_placed", "game_over_penalty", "hole_penalty",
               "center_bonus", "combo_multiplier_bonus", "survival_bonus")
REWARD_DEFAULTS = dict(line_clear_base=1.0, block_placed=0.01, game_over_penalty=-1.0,
                       hole_penalty=-0.05, center_bonus=0.02, combo_multiplier_bonus=0.5,
                       survival_bonus=0.001)   # reference block_blast_env.py:63-71

#: 32-byte record of bb_env_set_episode_end_buffer
EPISODE_END_DTYPE = np.dtype([("board", "<u8"), ("pieces", "<u4"), ("lines_total", "<i4"), ("max_streak", "<i4"),
                              ("blocks_total", "<i4"), ("holes_fill", "<u4"), ("last_move", "<u4")])

#: 48-byte per-env record of bb_env_get_state / bb_env_set_state
STATE_DTYPE = np.dtype([("board", "<u8"), ("pieces", "<u4"), ("aux", "<u4"), ("score", "<i4"),
                        ("streak", "<i4"), ("moves", "<i4"), ("lines_total", "<i4"),
                        ("max_streak", "<i4"), ("blocks_total", "<i4"), ("draw_ctr", "<u4"),
                        ("policy_ctr", "<u4")])

_lib = None


class BBGpuError(RuntimeError):
    pass


def lib():
    """The loaded library; raises if it has not been built (run ``python -m bbgpu.build`` or
    ``__graft_entry__.build()``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BBGpuError("libbbgpu.so not found at %s: the CUDA extension must be built "
                         "(python __graft_entry__.py build); there is no CPU fallback" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i64, u64, i32, u32 = C.c_void_p, C.c_int64, C.c_uint64, C.c_int32, C.c_uint32
    L.bb_version.restype = C.c_int
    L.bb_last_error.restype = C.c_char_p
    L.bb_piece_table.argtypes = [vp, vp, vp]
    L.bb_env_create.argtypes = [C.POINTER(vp), i64, u64, i64, vp, u32]
    L.bb_env_destroy.argtypes = [vp]
    L.bb_env_num_envs.argtypes = [vp]
    L.bb_env_num_envs.restype = i64
    L.bb_env_set_episode_end_buffer.argtypes = [vp, vp]
    L.bb_env_set_trios.argtypes = [vp, vp, i64, vp]
    L.bb_env_reset.argtypes = [vp, vp, vp, vp]
    L.bb_env_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.bb_env_step_random.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, vp]
    L.bb_env_rollout_random.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp]
    L.bb_env_observe.argtypes = [vp, vp, vp, vp, vp]
    L.bb_env_sample_valid_actions.argtypes = [vp, u64, vp, vp, vp]
    L.bb_env_expand.argtypes = [vp, u64, i32, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.bb_env_get_state.argtypes = [vp, vp, vp]
    L.bb_env_set_state.argtypes = [vp, vp, vp]
    L.bb_env_step_host.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.bb_env_fetch_step_info.argtypes = [vp, vp, vp, vp, vp]
    L.bb_env_host_dense_layout.argtypes = [i64, C.POINTER(i64), C.POINTER(i64)]
    L.bb_env_step_host_dense.argtypes = [vp, vp, vp, vp]
    L.bb_env_observe_host_dense.argtypes = [vp, vp, vp]
    L.bb_unpack_obs.argtypes = [vp, vp, vp, i64, vp, C.c_int, vp, C.c_int, i64, vp]
    L.bb_unpack_obs_reference_layout.argtypes = [vp, vp, vp, i64, vp, vp, vp, i64, vp]
    L.bb_gather_minibatch.argtypes = [vp, i64, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_int, vp, vp, vp, vp, vp, vp]
    L.bb_unpack_obs_sym.argtypes = [vp, vp, vp, vp, C.c_int, i64, vp]
    L.bb_sym_logits_mean.argtypes = [vp, C.c_int, vp, vp, i64, vp]
    L.bb_sym_logits_mean_backward.argtypes = [vp, vp, vp, C.c_int, i64, vp]
    L.bb_sym_canonical.argtypes = [vp, vp, vp, vp, vp, vp, i64, vp]
    L.bb_sym_logits_canonical.argtypes = [vp, C.c_int, vp, vp, vp, i64, vp]
    L.bb_sym_logits_canonical_backward.argtypes = [vp, vp, vp, vp, C.c_int, i64, vp]
    L.bb_masked_sample.argtypes = [vp, C.c_int, vp, i64, u64, u64, C.c_int, vp, vp, vp, i64, i64, vp, vp]
    L.bb_masked_head_backward.argtypes = [vp, C.c_int, vp, i64, vp, vp, vp, vp, i64, vp]
    L.bb_ppo_loss.argtypes = [vp, C.c_int, vp, i64, vp, vp, vp, vp, vp, C.c_double, C.c_double, C.c_double, vp, vp, vp, i64, vp]
    L.bb_env_host_layout.argtypes = [i64, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]
    L.bb_bn_workspace_size.restype = i64
    L.bb_bn_workspace_size.argtypes = [C.c_int]
    L.bb_bn_relu_forward.argtypes = [vp, vp, vp, vp, vp, vp, vp, C.c_double, C.c_double, C.c_int, vp, vp, vp, vp, i64, C.c_int, vp]
    L.bb_bn_relu_backward.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, C.c_int, vp]
    L.bb_bn_relu_backward_no_skip.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, C.c_int, vp]
    L.bb_gae.argtypes = [vp, vp, vp, vp, C.c_double, C.c_double, vp, vp, vp, i64, i64, vp]
    if L.bb_version() != ABI_VERSION:
        raise BBGpuError("libbbgpu.so ABI %d != expected %d" % (L.bb_version(), ABI_VERSION))
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise BBGpuError("libbbgpu: %s (code %d)" % (lib().bb_last_error().decode(), rc))


def ptr(t):
    """Device (or host) address of a torch tensor / numpy array / None."""
    if t is None:
        return None
    if isinstance(t, np.ndarray):
        return t.ctypes.data
    return t.data_ptr()


def current_stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def reward_cfg_array(reward_config=None):
    cfg = dict(REWARD_DEFAULTS)
    if reward_config:
        cfg.update(reward_config)
    return np.array([cfg[k] for k in REWARD_KEYS], dtype=np.float64)


def piece_table():
    masks = np.zeros(37, np.uint64)
    inb = np.zeros(37, np.uint64)
    nblk = np.zeros(37, np.uint8)
    check(lib().bb_piece_table(ptr(masks), ptr(inb), ptr(nblk)))
    return masks, inb, nblk


class EnvHandle:
    """Owns one ``bb_env`` on the current CUDA device."""

    def __init__(self, n_envs, seed=0, global_env_offset=0, reward_config=None, flags=0):
        import torch
        if not torch.cuda.is_available():
            raise BBGpuError("bbgpu needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.n = int(n_envs)
        self.device = torch.device("cuda", torch.cuda.current_device())
        h = C.c_void_p()
        cfg = reward_cfg_array(reward_config)
        check(lib().bb_env_create(C.byref(h), self.n, int(seed) & (2 ** 64 - 1), int(global_env_offset),
                                  ptr(cfg), int(flags)))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            lib().bb_env_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_episode_end_buffer(self, records):
        """records: CUDA uint8 tensor of n*32 bytes (or None); must outlive the handle's use of it."""
        self._ep_end_keepalive = records
        check(lib().bb_env_set_episode_end_buffer(self.h, ptr(records)))

    def set_trios(self, trios):
        """Injected candidate trios (replay / parity mode): uint8 array [n, L, 3] of piece indices,
        or None to return to the Philox streams.  Call reset() afterwards."""
        if trios is None:
            check(lib().bb_env_set_trios(self.h, None, 0, current_stream()))
            return
        t = np.ascontiguousarray(trios, dtype=np.uint8)
        assert t.ndim == 3 and t.shape[0] == self.n and t.shape[2] == 3, t.shape
        check(lib().bb_env_set_trios(self.h, ptr(t), t.shape[1], current_stream()))

    def reset(self, reset_mask=None, mask_out=None):
        check(lib().bb_env_reset(self.h, ptr(reset_mask), ptr(mask_out), current_stream()))

    def step(self, actions, rewards, terminated, mask_out=None, ep_score=None, ep_len=None, info_out=None,
             board_out=None, pieces_out=None, stats=None):
        check(lib().bb_env_step(self.h, ptr(actions), ptr(rewards), ptr(terminated), ptr(mask_out), ptr(board_out),
                                ptr(pieces_out), ptr(ep_score), ptr(ep_len), ptr(info_out), ptr(stats), current_stream()))

    def step_random(self, n_steps=1, actions_out=None, rewards=None, terminated=None, mask_out=None, stats=None,
                    mask_in=None):
        check(lib().bb_env_step_random(self.h, int(n_steps), ptr(actions_out), ptr(rewards), ptr(terminated),
                                       ptr(mask_out), ptr(stats), ptr(mask_in), current_stream()))

    def rollout_random(self, n_steps, actions_out=None, rewards=None, terminated=None, mask_out=None, stats=None):
        """n_steps in one launch, outputs of EVERY step written to [n_steps, ...] arrays."""
        check(lib().bb_env_rollout_random(self.h, int(n_steps), ptr(actions_out), ptr(rewards), ptr(terminated),
                                          ptr(mask_out), ptr(stats), current_stream()))

    def sample_valid_actions(self, call_counter, actions_out=None, h_actions_out=None):
        check(lib().bb_env_sample_valid_actions(self.h, int(call_counter), ptr(actions_out), ptr(h_actions_out),
                                                current_stream()))

    def observe(self, board_out=None, pieces_out=None, mask_out=None):
        check(lib().bb_env_observe(self.h, ptr(board_out), ptr(pieces_out), ptr(mask_out), current_stream()))

    def expand(self, call_counter, samples=1):
        """One-ply successors of every env's current state (bb_env_expand; no state changes).
        Two calls: a size query, then the fill with the same ``call_counter`` (the item count is read
        back, which synchronises the stream).  Returns CUDA tensors: ``offsets`` int64 [n+1] (items of
        env i are offsets[i]:offsets[i+1]), ``action`` int32, ``reward`` f32, ``terminated`` u8,
        ``info`` int32 (the u32 info word), ``board`` int64, ``pieces`` int32 — all [items] — and
        ``mask`` int64 [3, items]."""
        import torch
        dev = self.device
        offsets = torch.empty(self.n + 1, dtype=torch.int64, device=dev)
        L = lib()
        check(L.bb_env_expand(self.h, int(call_counter), int(samples), 0, ptr(offsets), None, None, None, None, None,
                              None, None, current_stream()))
        cap = int(offsets[self.n].item())
        out = {"offsets": offsets,
               "action": torch.empty(cap, dtype=torch.int32, device=dev),
               "reward": torch.empty(cap, dtype=torch.float32, device=dev),
               "terminated": torch.empty(cap, dtype=torch.uint8, device=dev),
               "info": torch.empty(cap, dtype=torch.int32, device=dev),
               "board": torch.empty(cap, dtype=torch.int64, device=dev),
               "pieces": torch.empty(cap, dtype=torch.int32, device=dev),
               "mask": torch.empty((3, cap), dtype=torch.int64, device=dev)}
        check(L.bb_env_expand(self.h, int(call_counter), int(samples), cap, ptr(offsets), ptr(out["action"]),
                              ptr(out["reward"]), ptr(out["terminated"]), ptr(out["info"]), ptr(out["board"]),
                              ptr(out["pieces"]), ptr(out["mask"]), current_stream()))
        return out

    def get_state(self):
        rec = np.zeros(self.n, STATE_DTYPE)
        check(lib().bb_env_get_state(self.h, ptr(rec), current_stream()))
        return rec

    def set_state(self, rec):
        rec = np.ascontiguousarray(rec, dtype=STATE_DTYPE)
        assert rec.shape == (self.n,)
        check(lib().bb_env_set_state(self.h, ptr(rec), current_stream()))

    def step_host(self, actions, rewards, terminated, board=None, pieces=None, mask=None, ep_score=None, ep_len=None,
                  info=None):
        check(lib().bb_env_step_host(self.h, ptr(actions), ptr(rewards), ptr(terminated), ptr(board), ptr(pieces),
                                     ptr(mask), ptr(ep_score), ptr(ep_len), ptr(info), current_stream()))

    def fetch_step_info(self, ep_score=None, ep_len=None, info=None):
        """ep_score / ep_len / info arrays of the LAST host-buffer step (host buffers)."""
        check(lib().bb_env_fetch_step_info(self.h, ptr(ep_score), ptr(ep_len), ptr(info), current_stream()))

    def step_host_dense(self, actions, block):
        """Host-buffer step returning the reference's dense observation layout in one pinned block."""
        check(lib().bb_env_step_host_dense(self.h, ptr(actions), ptr(block), current_stream()))

    def observe_host_dense(self, block):
        check(lib().bb_env_observe_host_dense(self.h, ptr(block), current_stream()))


HOST_LAYOUT_FIELDS = ("mask", "board", "rewards", "pieces", "ep_score", "ep_len", "info", "term")


def host_layout(n_envs):
    """({field: byte offset}, total bytes) of the single-block result layout of bb_env_step_host
    (mask/board/rewards/pieces/term form the per-step prefix, ep_score/ep_len/info the tail)."""
    offs = (C.c_int64 * 8)()
    total, prefix = C.c_int64(), C.c_int64()
    check(lib().bb_env_host_layout(int(n_envs), offs, C.byref(total), C.byref(prefix)))
    return dict(zip(HOST_LAYOUT_FIELDS, [int(o) for o in offs])), int(total.value)


DENSE_LAYOUT_FIELDS = ("board", "pieces", "action_mask", "rewards", "term")


def pinned_dense_block(n_envs):
    """One pinned host block in the layout of bb_env_step_host_dense as typed torch views: board f32
    [n,8,8], pieces f32 [n,3,8,8], action_mask int8 [n,192], rewards f32 [n], term u8 [n]."""
    import torch
    offs = (C.c_int64 * 5)()
    total = C.c_int64()
    n = int(n_envs)
    check(lib().bb_env_host_dense_layout(n, offs, C.byref(total)))
    block = torch.zeros(int(total.value), dtype=torch.uint8).pin_memory()
    o = [int(x) for x in offs]
    return {"_block": block,
            "board": block[o[0]:o[1]].view(torch.float32).view(n, 8, 8),
            "pieces": block[o[1]:o[2]].view(torch.float32).view(n, 3, 8, 8),
            "action_mask": block[o[2]:o[3]].view(torch.int8).view(n, 192),
            "rewards": block[o[3]:o[4]].view(torch.float32),
            "term": block[o[4]:o[4] + n]}


def pinned_result_block(n_envs):
    """One pinned host block laid out for bb_env_step_host, as a dict of typed torch views
    (mask int64 [3,n], board int64, rewards f32, pieces int32, ep_score, ep_len, info int32, term u8)."""
    import torch
    offs, total = host_layout(n_envs)
    block = torch.zeros(total, dtype=torch.uint8).pin_memory()
    n = int(n_envs)
    dt = dict(mask=(torch.int64, 3 * n), board=(torch.int64, n), rewards=(torch.float32, n), pieces=(torch.int32, n),
              ep_score=(torch.int32, n), ep_len=(torch.int32, n), info=(torch.int32, n), term=(torch.uint8, n))
    out = {"_block": block}
    for k, (t, cnt) in dt.items():
        nbytes = cnt * torch.empty(0, dtype=t).element_size()
        out[k] = block[offs[k]:offs[k] + nbytes].view(t)
    out["mask"] = out["mask"].view(3, n)
    return out


def unpack_obs(board, pieces, mask, mask_stride, obs=None, mask_dense=None, n=None):
    import torch
    n = int(board.numel() if n is None else n)
    obs_dt = BB_BF16 if (obs is not None and obs.dtype == torch.bfloat16) else BB_F32
    mask_dt = BB_F32 if (mask_dense is not None and mask_dense.dtype == torch.float32) else BB_U8
    check(lib().bb_unpack_obs(ptr(board), ptr(pieces), ptr(mask), int(mask_stride), ptr(obs), obs_dt,
                              ptr(mask_dense), mask_dt, n, current_stream()))


def unpack_obs_reference_layout(board, pieces, mask, mask_stride, board_f32, pieces_f32, action_mask_i8=None, n=None):
    n = int(board.numel() if n is None else n)
    check(lib().bb_unpack_obs_reference_layout(ptr(board), ptr(pieces), ptr(mask), int(mask_stride), ptr(board_f32),
                                               ptr(pieces_f32), ptr(action_mask_i8), n, current_stream()))


def unpack_obs_sym(board, pieces, obs, index=None, n=None):
    """K7a (bb_unpack_obs_sym): obs [8n,4,8,8] f32 / bf16, row g*n + i = view g of packed row i (or index[i])."""
    import torch
    n = int((index.numel() if index is not None else board.numel()) if n is None else n)
    assert obs.is_contiguous() and obs.shape[0] == 8 * n
    dt = BB_BF16 if obs.dtype == torch.bfloat16 else BB_F32
    check(lib().bb_unpack_obs_sym(ptr(board), ptr(pieces), ptr(index), ptr(obs), dt, n, current_stream()))


def sym_logits_mean(logits, pieces, out):
    """K7b forward (bb_sym_logits_mean): logits [8n,192] f32 / bf16, pieces int32 [n] -> out f32 [n,192]."""
    import torch
    n = pieces.numel()
    assert logits.is_contiguous() and logits.shape == (8 * n, 192) and out.dtype == torch.float32 and out.is_contiguous()
    dt = BB_BF16 if logits.dtype == torch.bfloat16 else BB_F32
    check(lib().bb_sym_logits_mean(ptr(logits), dt, ptr(pieces), ptr(out), n, current_stream()))


def sym_logits_mean_backward(grad_out, pieces, grad_logits):
    """K7b backward (bb_sym_logits_mean_backward): grad_out f32 [n,192] -> grad_logits [8n,192] f32 / bf16."""
    import torch
    n = pieces.numel()
    assert grad_out.is_contiguous() and grad_out.dtype == torch.float32 and grad_logits.shape == (8 * n, 192)
    dt = BB_BF16 if grad_logits.dtype == torch.bfloat16 else BB_F32
    check(lib().bb_sym_logits_mean_backward(ptr(grad_out), ptr(pieces), ptr(grad_logits), dt, n, current_stream()))


def sym_canonical(board, pieces, board_out, pieces_out, views_out, index=None, n=None):
    """K7c (bb_sym_canonical): canonical view board_out int64 [n] / pieces_out int32 [n] and view set views_out
    uint8 [n] of packed row i (or index[i])."""
    n = int((index.numel() if index is not None else board.numel()) if n is None else n)
    assert board_out.numel() >= n and pieces_out.numel() >= n and views_out.numel() >= n
    check(lib().bb_sym_canonical(ptr(board), ptr(pieces), ptr(index), ptr(board_out), ptr(pieces_out), ptr(views_out), n,
                                 current_stream()))


def sym_logits_canonical(logits, pieces, views, out):
    """K7c forward (bb_sym_logits_canonical): canonical-row logits [n,192] f32 / bf16, the states' own pieces int32
    [n] and view sets uint8 [n] -> out f32 [n,192] in the states' frames."""
    import torch
    n = pieces.numel()
    assert logits.is_contiguous() and logits.shape == (n, 192) and out.dtype == torch.float32 and out.is_contiguous()
    assert views.numel() == n and views.dtype == torch.uint8
    dt = BB_BF16 if logits.dtype == torch.bfloat16 else BB_F32
    check(lib().bb_sym_logits_canonical(ptr(logits), dt, ptr(pieces), ptr(views), ptr(out), n, current_stream()))


def sym_logits_canonical_backward(grad_out, pieces, views, grad_logits):
    """K7c backward (bb_sym_logits_canonical_backward): grad_out f32 [n,192] -> grad_logits [n,192] f32 / bf16."""
    import torch
    n = pieces.numel()
    assert grad_out.is_contiguous() and grad_out.dtype == torch.float32 and grad_logits.shape == (n, 192)
    assert views.numel() == n and views.dtype == torch.uint8
    dt = BB_BF16 if grad_logits.dtype == torch.bfloat16 else BB_F32
    check(lib().bb_sym_logits_canonical_backward(ptr(grad_out), ptr(pieces), ptr(views), ptr(grad_logits), dt, n,
                                                 current_stream()))


def gather_minibatch(index, n_envs, board, pieces, mask, action, logp, adv, ret, adv_mean_std, obs, mask_out,
                     action_out, logp_out, adv_out, ret_out):
    """RolloutBuffer.get_samples' gathers + K2 in one call (bb_gather_minibatch); obs None: no planes."""
    import torch
    dt = BB_BF16 if obs is not None and obs.dtype == torch.bfloat16 else BB_F32
    check(lib().bb_gather_minibatch(ptr(index), int(index.numel()), int(n_envs), ptr(board), ptr(pieces), ptr(mask),
                                    ptr(action), ptr(logp), ptr(adv), ptr(ret), ptr(adv_mean_std), ptr(obs), dt,
                                    ptr(mask_out), ptr(action_out), ptr(logp_out), ptr(adv_out), ptr(ret_out),
                                    current_stream()))


def masked_sample(logits, mask, mask_stride, seed, call_counter, mode, action, logp=None, entropy=None,
                  row_offset=0, call_counter_dev=None):
    import torch
    n = logits.shape[0]
    assert logits.is_contiguous() and logits.shape[1] == 192
    dt = BB_BF16 if logits.dtype == torch.bfloat16 else BB_F32
    check(lib().bb_masked_sample(ptr(logits), dt, ptr(mask), int(mask_stride), int(seed) & (2 ** 64 - 1),
                                 int(call_counter), int(mode), ptr(action), ptr(logp), ptr(entropy), n,
                                 int(row_offset), ptr(call_counter_dev), current_stream()))


def masked_head_backward(logits, mask, mask_stride, action, grad_logp, grad_entropy, grad_logits):
    import torch
    n = logits.shape[0]
    dt = BB_BF16 if logits.dtype == torch.bfloat16 else BB_F32
    check(lib().bb_masked_head_backward(ptr(logits), dt, ptr(mask), int(mask_stride), ptr(action), ptr(grad_logp),
                                        ptr(grad_entropy), ptr(grad_logits), n, current_stream()))


def ppo_loss(logits, mask, mask_stride, action, old_logp, adv, ret, values, clip, value_coef, entropy_coef,
             grad_logits, grad_values, sums5):
    import torch
    n = logits.shape[0]
    dt = BB_BF16 if logits.dtype == torch.bfloat16 else BB_F32
    check(lib().bb_ppo_loss(ptr(logits), dt, ptr(mask), int(mask_stride), ptr(action), ptr(old_logp), ptr(adv), ptr(ret),
                            ptr(values), float(clip), float(value_coef), float(entropy_coef), ptr(grad_logits),
                            ptr(grad_values), ptr(sums5), n, current_stream()))


def bn_workspace_size(channels):
    n = int(lib().bb_bn_workspace_size(int(channels)))
    if n < 0:
        raise BBGpuError("bb_bn_workspace_size: unsupported channel count %d" % channels)
    return n


def bn_relu_forward(x, skip, gamma, beta, pre_bias, running_mean, running_var, momentum, eps, training, y, save_mean,
                    save_rstd, workspace, rows, channels):
    check(lib().bb_bn_relu_forward(ptr(x), ptr(skip), ptr(gamma), ptr(beta), ptr(pre_bias), ptr(running_mean), ptr(running_var),
                                   float(momentum), float(eps), int(bool(training)), ptr(y), ptr(save_mean), ptr(save_rstd),
                                   ptr(workspace), int(rows), int(channels), current_stream()))


def bn_relu_backward(x, y, grad_y, gamma, save_mean, save_rstd, grad_x, grad_skip, grad_gamma, grad_beta, workspace,
                     rows, channels):
    check(lib().bb_bn_relu_backward(ptr(x), ptr(y), ptr(grad_y), ptr(gamma), ptr(save_mean), ptr(save_rstd), ptr(grad_x),
                                    ptr(grad_skip), ptr(grad_gamma), ptr(grad_beta), ptr(workspace), int(rows), int(channels),
                                    current_stream()))


def bn_relu_backward_no_skip(x, grad_y, gamma, beta, save_mean, save_rstd, grad_x, grad_gamma, grad_beta, workspace, rows,
                             channels):
    check(lib().bb_bn_relu_backward_no_skip(ptr(x), ptr(grad_y), ptr(gamma), ptr(beta), ptr(save_mean), ptr(save_rstd),
                                            ptr(grad_x), ptr(grad_gamma), ptr(grad_beta), ptr(workspace), int(rows),
                                            int(channels), current_stream()))


def gae(rewards, values, dones, last_values, gamma, lam, adv, ret, moments=None):
    T, N = rewards.shape
    check(lib().bb_gae(ptr(rewards), ptr(values), ptr(dones), ptr(last_values), float(gamma), float(lam),
                       ptr(adv), ptr(ret), ptr(moments), T, N, current_stream()))
