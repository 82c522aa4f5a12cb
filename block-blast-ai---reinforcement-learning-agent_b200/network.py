"""Policy/value network with the reference's architecture and state_dict layout.

Mirror of ``BlockBlastNetwork`` (reference src/models/network.py:34-271): 4 input planes
(board + 3 piece masks) -> conv 64 -> conv 128 + residual block -> conv 128 + residual block
-> FC 8192->512->256 (ReLU, Dropout 0.1) -> policy head 256->256->192, value head 256->128->1;
5,290,113 parameters.  Module and parameter names are the reference's, so checkpoints written
by either side load in the other (``network_state_dict``, src/agents/ppo.py:425-439).

The CNN body stays PyTorch (north_star).  What is replaced is the categorical head:
``get_action_and_value`` without gradients (rollout / evaluation) runs the fused K3 kernel
(-inf masking + softmax + sample/argmax + log-prob + masked entropy, network.py:172-262);
with gradients (given actions) the same maths is expressed in torch ops so autograd applies.
The PPO update runs the whole loss tail after the CNN as one kernel (``PPOLossTail``).
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import capi


_BN_WORKSPACE = {}


def _bn_workspace(channels, device):
    key = (device.index, channels)
    ws = _BN_WORKSPACE.get(key)
    if ws is None:
        ws = _BN_WORKSPACE[key] = torch.empty(capi.bn_workspace_size(channels), dtype=torch.float32, device=device)
    return ws


class FusedBNReLU(torch.autograd.Function):
    """relu(BatchNorm2d(x) (+ skip)) on channels-last bf16 activations as HBM-roofline passes
    (bb_bn_relu_forward / bb_bn_relu_backward) instead of torch's batch_norm + add + relu kernels;
    the module keeps its nn.BatchNorm2d parameters and buffers (running statistics are updated in
    place exactly like torch: momentum, unbiased variance)."""

    @staticmethod
    def forward(ctx, x, skip, weight, bias, running_mean, running_var, training, momentum, eps, pre_bias=None):
        x = x.contiguous(memory_format=torch.channels_last)
        n, c, h, w = x.shape
        rows = n * h * w
        if skip is not None:
            skip = skip.to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
        y = torch.empty_like(x)
        save_mean = torch.empty(c, dtype=torch.float32, device=x.device)
        save_rstd = torch.empty(c, dtype=torch.float32, device=x.device)
        pb = None if pre_bias is None else pre_bias.detach().float().contiguous()
        capi.bn_relu_forward(x, skip, weight, bias, pb, running_mean, running_var, momentum, eps, training, y,
                             save_mean, save_rstd, _bn_workspace(c, x.device), rows, c)
        ctx.has_skip = skip is not None
        # without a residual input the ReLU mask is recomputed from x in backward: y need not be kept for it
        if ctx.has_skip:
            ctx.save_for_backward(x, y, weight, save_mean, save_rstd)
        else:
            ctx.save_for_backward(x, bias.detach(), weight, save_mean, save_rstd)
        return y

    @staticmethod
    def backward(ctx, grad_y):
        x, y_or_beta, weight, save_mean, save_rstd = ctx.saved_tensors
        n, c, h, w = x.shape
        grad_y = grad_y.to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
        grad_x = torch.empty_like(x)
        grad_skip = torch.empty_like(x) if ctx.has_skip else None
        grad_gamma = torch.empty(c, dtype=torch.float32, device=x.device)
        grad_beta = torch.empty(c, dtype=torch.float32, device=x.device)
        if ctx.has_skip:
            capi.bn_relu_backward(x, y_or_beta, grad_y, weight, save_mean, save_rstd, grad_x, grad_skip, grad_gamma, grad_beta,
                                  _bn_workspace(c, x.device), n * h * w, c)
        else:
            capi.bn_relu_backward_no_skip(x, grad_y, weight, y_or_beta, save_mean, save_rstd, grad_x, grad_gamma, grad_beta,
                                          _bn_workspace(c, x.device), n * h * w, c)
        return grad_x, grad_skip, grad_gamma, grad_beta, None, None, None, None, None, None


def _bn_fusable(bn, channels):
    return (channels % 8 == 0 and bn.affine and bn.track_running_stats and bn.momentum is not None
            and (bn.training or not torch.is_grad_enabled()))


def bn_relu(bn, x, skip=None, fused=False, pre_bias=None):
    """relu(bn(x) (+ skip)); the fused kernels when asked for and applicable (CUDA, bf16, channel
    count a multiple of 8, affine BatchNorm with running statistics, training mode or no autograd).
    ``pre_bias``: conv bias the caller left out of x (see conv_bn_relu)."""
    if fused and x.is_cuda and x.dtype == torch.bfloat16 and x.dim() == 4 and _bn_fusable(bn, x.shape[1]):
        if bn.training:
            bn.num_batches_tracked.add_(1)
        return FusedBNReLU.apply(x, skip, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.training,
                                 bn.momentum, bn.eps, pre_bias)
    if pre_bias is not None:
        x = x + pre_bias.to(x.dtype).view(1, -1, 1, 1)
    y = bn(x)
    if skip is not None:
        y = y + skip
    return F.relu(y)


def conv_bn_relu(conv, bn, x, skip=None, fused=False):
    """relu(bn(conv(x)) (+ skip)).  On the fused path the convolution runs WITHOUT its bias:
    BatchNorm subtracts the batch mean, so a per-channel constant in front of it cancels exactly in
    the output and its gradient is identically zero; the bias is handed to the BatchNorm kernel,
    which keeps it in the tracked running mean (and applies it in eval mode).  This removes the
    bias-add and bias-gradient passes over the activations (15 % and 9 % of the CNN's time)."""
    if (fused and x.is_cuda and conv.bias is not None and _bn_fusable(bn, conv.out_channels)
            and torch.is_autocast_enabled() and torch.get_autocast_dtype("cuda") == torch.bfloat16):
        y = F.conv2d(x, conv.weight, None, conv.stride, conv.padding, conv.dilation, conv.groups)
        return bn_relu(bn, y, skip, True, conv.bias)
    return bn_relu(bn, conv(x), skip, fused)


class ResidualBlock(nn.Module):
    """conv-bn-relu-conv-bn + skip, relu (reference network.py:14-31)."""
    fused_bn = False

    def __init__(self, channels):
        super().__init__()
        self.conv1 = nn.Conv2d(channels, channels, 3, padding=1)
        self.bn1 = nn.BatchNorm2d(channels)
        self.conv2 = nn.Conv2d(channels, channels, 3, padding=1)
        self.bn2 = nn.BatchNorm2d(channels)

    def forward(self, x):
        y = conv_bn_relu(self.conv1, self.bn1, x, None, self.fused_bn)
        return conv_bn_relu(self.conv2, self.bn2, y, x, self.fused_bn)


def _pack_mask_planes(mask_dense):
    """(B,192) 0/1 tensor -> int64 [3,B] bit planes (bit = row*8+col), on the mask's device."""
    b = mask_dense.shape[0]
    bits = (mask_dense != 0).reshape(b, 3, 8, 8).to(torch.int64)
    byte_w = (2 ** torch.arange(8, device=mask_dense.device, dtype=torch.int64)).view(1, 1, 1, 8)
    rows = (bits * byte_w).sum(-1)                                   # (B,3,8) row bytes 0..255
    shifts = (8 * torch.arange(8, device=mask_dense.device, dtype=torch.int64)).view(1, 1, 8)
    hi_fix = rows << shifts                                          # row 7 lands in the sign bit: two's complement is fine
    return hi_fix.sum(-1).t().contiguous()                           # wraps modulo 2**64


class PPOLossTail(torch.autograd.Function):
    """The whole loss tail of PPOAgent.update (src/agents/ppo.py:366-395) as ONE kernel
    (bb_ppo_loss, SURVEY §8f item 2): forward returns the scalar loss and the five metric means
    (policy_loss, value_loss, entropy, approx_kl, clip_fraction); the gradients w.r.t. logits and
    values are produced by the same pass and only scaled in backward."""

    @staticmethod
    def forward(ctx, logits, values, planes, action, old_logp, adv, ret, clip, value_coef, entropy_coef):
        lg = logits.detach()
        if lg.dtype not in (torch.float32, torch.bfloat16):
            lg = lg.float()
        lg = lg.contiguous()
        n = lg.shape[0]
        v = values.detach().float().contiguous()
        g_logits = torch.empty_like(lg)
        g_values = torch.empty(n, dtype=torch.float32, device=lg.device)
        sums = torch.zeros(5, dtype=torch.float64, device=lg.device)
        capi.ppo_loss(lg, planes, planes.stride(0), action.to(torch.int32).contiguous(), old_logp.float().contiguous(),
                      adv.float().contiguous(), ret.float().contiguous(), v, clip, value_coef, entropy_coef,
                      g_logits, g_values, sums)
        means = sums / n
        loss = (means[0] + value_coef * means[1] - entropy_coef * means[2]).float()
        ctx.save_for_backward(g_logits, g_values)
        ctx.dtypes = (logits.dtype, values.dtype)
        ctx.mark_non_differentiable(means)
        return loss, means

    @staticmethod
    def backward(ctx, g_loss, _g_means):
        g_logits, g_values = ctx.saved_tensors
        return ((g_logits * g_loss).to(ctx.dtypes[0]), (g_values * g_loss).to(ctx.dtypes[1]),
                None, None, None, None, None, None, None, None)


class SymmetryMean(torch.autograd.Function):
    """Group average of the policy logits over the eight board symmetries (K7b, bb_sym_logits_mean): raw
    logits [8n,192] of the eight views (rows g*n + i, as bb_unpack_obs_sym writes the observations) and the
    pieces words int32 [n] of the states -> f32 [n,192] logits of the states, 0 at positions that are always
    masked.  The backward pass is the kernel's transposed map, in the logits' dtype."""

    @staticmethod
    def forward(ctx, logits, pieces):
        lg = logits.detach()
        if lg.dtype not in (torch.float32, torch.bfloat16):
            lg = lg.float()
        lg = lg.contiguous()
        out = torch.empty((pieces.numel(), 192), dtype=torch.float32, device=lg.device)
        capi.sym_logits_mean(lg, pieces, out)
        ctx.save_for_backward(pieces)
        ctx.dtype = lg.dtype
        return out

    @staticmethod
    def backward(ctx, g):
        pieces, = ctx.saved_tensors
        grad = torch.empty((8 * pieces.numel(), 192), dtype=ctx.dtype, device=g.device)
        capi.sym_logits_mean_backward(g.float().contiguous(), pieces, grad)
        return grad, None


class CanonicalFrame(torch.autograd.Function):
    """The canonical-frame policy's logit map (K7c, bb_sym_logits_canonical): raw logits [n,192] of the
    canonical views (bb_sym_canonical), the states' own pieces words int32 [n] and view sets uint8 [n] -> f32
    [n,192] logits in the states' own frames, 0 at positions that are always masked.  The backward pass is
    the kernel's transposed map, in the logits' dtype."""

    @staticmethod
    def forward(ctx, logits, pieces, views):
        lg = logits.detach()
        if lg.dtype not in (torch.float32, torch.bfloat16):
            lg = lg.float()
        lg = lg.contiguous()
        out = torch.empty((pieces.numel(), 192), dtype=torch.float32, device=lg.device)
        capi.sym_logits_canonical(lg, pieces, views, out)
        ctx.save_for_backward(pieces, views)
        ctx.dtype = lg.dtype
        return out

    @staticmethod
    def backward(ctx, g):
        pieces, views = ctx.saved_tensors
        grad = torch.empty((pieces.numel(), 192), dtype=ctx.dtype, device=g.device)
        capi.sym_logits_canonical_backward(g.float().contiguous(), pieces, views, grad)
        return grad, None, None


class BlockBlastNetwork(nn.Module):
    def __init__(self, board_size=8, num_pieces=3, conv_channels=(64, 128, 128), fc_hidden=(512, 256),
                 action_space_size=192, use_residual=True, use_batch_norm=True):
        super().__init__()
        self.board_size, self.num_pieces, self.action_space_size = board_size, num_pieces, action_space_size
        layers, cin = [], 1 + num_pieces
        for i, cout in enumerate(conv_channels):
            layers.append(nn.Conv2d(cin, cout, 3, padding=1))
            if use_batch_norm:
                layers.append(nn.BatchNorm2d(cout))
            layers.append(nn.ReLU())
            if use_residual and i > 0:
                layers.append(ResidualBlock(cout))
            cin = cout
        self.conv_encoder = nn.Sequential(*layers)
        fc, fin = [], conv_channels[-1] * board_size * board_size
        for h in fc_hidden:
            fc += [nn.Linear(fin, h), nn.ReLU(), nn.Dropout(0.1)]
            fin = h
        self.fc_encoder = nn.Sequential(*fc)
        self.policy_head = nn.Sequential(nn.Linear(fin, 256), nn.ReLU(), nn.Linear(256, action_space_size))
        self.value_head = nn.Sequential(nn.Linear(fin, 128), nn.ReLU(), nn.Linear(128, 1))
        # categorical sampling noise (K3, Philox SAMPLE stream): keyed by (sample_seed, global row id =
        # sample_row_offset + row, call counter).  The counter lives on the device so that a captured
        # CUDA graph advances it on every replay; it is not a registered buffer (the state_dict stays the
        # reference's) — PPOAgent.save / load carry it.
        self.sample_seed = 0
        self.sample_row_offset = 0
        self._sample_counter = None
        for m in self.modules():                      # reference network.py:122-133
            if isinstance(m, (nn.Linear, nn.Conv2d)):
                nn.init.kaiming_uniform_(m.weight, nonlinearity="relu")
                if m.bias is not None:
                    nn.init.zeros_(m.bias)

    # ---------------------------------------------------------------- body
    def set_fused_bn(self, on=True):
        """Route every BatchNorm2d + ReLU (+ residual add) of the encoder through FusedBNReLU."""
        self.fused_bn = bool(on)
        for m in self.modules():
            if isinstance(m, ResidualBlock):
                m.fused_bn = bool(on)
        return self

    def _encode(self, x):
        if not getattr(self, "fused_bn", False):
            return self.conv_encoder(x)
        mods = list(self.conv_encoder)
        i = 0
        while i < len(mods):
            m = mods[i]
            if (isinstance(m, nn.Conv2d) and i + 2 < len(mods) and isinstance(mods[i + 1], nn.BatchNorm2d)
                    and isinstance(mods[i + 2], nn.ReLU)):
                x = conv_bn_relu(m, mods[i + 1], x, None, True)
                i += 3
            elif isinstance(m, nn.BatchNorm2d) and i + 1 < len(mods) and isinstance(mods[i + 1], nn.ReLU):
                x = bn_relu(m, x, None, True)
                i += 2
            else:
                x = m(x)
                i += 1
        return x

    def _flatten_fc(self, x):
        """fc_encoder(x.flatten(1)).  The first Linear's weight is laid out for the NCHW flatten
        (state_dict compatibility); for channels-last activations x.flatten(1) is a 2 x 0.5 GB
        transposing copy per 32,768-sample minibatch (forward + backward), so the 8 MB weight is
        permuted to (h, w, c) order instead and the activations are used as they lie in memory."""
        fc0 = self.fc_encoder[0]
        if (getattr(self, "fused_bn", False) and x.dim() == 4 and isinstance(fc0, nn.Linear)
                and x.is_contiguous(memory_format=torch.channels_last) and not x.is_contiguous()):
            b, c, h, w = x.shape
            flat = x.permute(0, 2, 3, 1).reshape(b, h * w * c)                                  # a view
            wperm = fc0.weight.view(fc0.out_features, c, h, w).permute(0, 2, 3, 1).reshape(fc0.out_features, h * w * c)
            y = F.linear(flat, wperm, fc0.bias)
            for m in list(self.fc_encoder)[1:]:
                y = m(y)
            return y
        return self.fc_encoder(x.flatten(1))

    def trunk(self, x):
        """x: (B,4,8,8) = cat([board, pieces]) (network.py:152-158) -> (raw logits (B,192), value (B,))."""
        x = self._encode(x)
        x = self._flatten_fc(x)
        return self.policy_head(x), self.value_head(x).squeeze(-1)

    @staticmethod
    def _nchw(board, pieces):
        if board.dim() == 3:
            board = board.unsqueeze(1)
        return torch.cat([board, pieces], dim=1)

    def forward(self, board, pieces, action_mask=None):
        logits, value = self.trunk(self._nchw(board, pieces))
        if action_mask is not None:                    # network.py:172-180
            logits = logits.masked_fill(~action_mask.bool(), float("-inf"))
        return logits, value

    def get_value(self, board, pieces):
        return self.forward(board, pieces)[1]

    # ---------------------------------------------------------------- masked categorical head
    def sample_counter(self, device=None):
        """int64[1] CUDA tensor: number of sampling calls made so far."""
        if self._sample_counter is None or (device is not None and self._sample_counter.device != torch.device(device)):
            dev = device if device is not None else next(self.parameters()).device
            old = 0 if self._sample_counter is None else int(self._sample_counter.item())
            self._sample_counter = torch.full((1,), old, dtype=torch.int64, device=dev)
        return self._sample_counter

    @property
    def sample_calls(self):
        return 0 if self._sample_counter is None else int(self._sample_counter.item())

    @sample_calls.setter
    def sample_calls(self, value):
        self.sample_counter().fill_(int(value))

    def head_from_logits(self, raw_logits, mask_planes, action=None, deterministic=False, need_entropy=True):
        """K3 on raw (unmasked) logits and packed mask planes int64 [3,B]; no autograd."""
        n = raw_logits.shape[0]
        logits = raw_logits.detach()
        if logits.dtype not in (torch.float32, torch.bfloat16):
            logits = logits.float()
        logits = logits.contiguous()
        logp = torch.empty(n, dtype=torch.float32, device=logits.device)
        ent = torch.empty(n, dtype=torch.float32, device=logits.device) if need_entropy else None
        if action is None:
            act = torch.empty(n, dtype=torch.int32, device=logits.device)
            ctr = self.sample_counter(logits.device)
            capi.masked_sample(logits, mask_planes, mask_planes.stride(0), self.sample_seed, 1,
                               1 if deterministic else 0, act, logp, ent, self.sample_row_offset, ctr)
            if not deterministic:
                ctr.add_(1)
        else:
            act = action.to(torch.int32).contiguous()
            capi.masked_sample(logits, mask_planes, mask_planes.stride(0), 0, 0, 2, act, logp, ent)
        return act, logp, ent

    def get_action_and_value(self, board, pieces, action_mask, action=None, deterministic=False):
        """network.py:184-230.  Returns (action int64, log_prob, entropy, value)."""
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()) and action is not None:
            return self.evaluate_actions(self._nchw(board, pieces), action_mask, action)
        logits, value = self.trunk(self._nchw(board, pieces))
        if not logits.is_cuda:
            raise capi.BBGpuError("BlockBlastNetwork's masked head runs on CUDA only (no CPU fallback)")
        planes = _pack_mask_planes(action_mask)
        act, logp, ent = self.head_from_logits(logits, planes, action, deterministic)
        return act.long(), logp, ent, value

    def evaluate_actions(self, x_nchw, action_mask, action):
        """Differentiable log-prob / masked entropy of given actions (PPO update,
        src/agents/ppo.py:366-369 -> network.py:210-262), same formulas as K3."""
        logits, value = self.trunk(x_nchw)
        logits = logits.float()
        valid = action_mask.bool()
        probs = F.softmax(logits.masked_fill(~valid, float("-inf")), dim=-1)
        eps = torch.finfo(torch.float32).eps
        pn = probs / probs.sum(-1, keepdim=True)
        logp = torch.log(pn.clamp(eps, 1 - eps)).gather(1, action.long().unsqueeze(1)).squeeze(1)
        q = probs / probs.sum(-1, keepdim=True).clamp(min=1e-10)      # probs already 0 where masked
        ent = -(q * torch.log(q.clamp(min=1e-10)) * valid).sum(-1)
        return action, logp, ent, value
