// bb_policy_kernels.cu — K2 (packed obs -> dense NCHW planes / dense mask) and K3 (fused
// -inf masking + softmax + categorical sample + log-prob + masked entropy) for sm_100a.
//
// K2 replaces engine.get_observation + Piece.to_mask (src/game/engine.py:489-507,
// src/game/pieces.py:39-45) and the torch.cat at src/models/network.py:152-158:
// 36 B in, 1,024 B (f32) / 512 B (bf16) out per env; a warp writes one env's 4x8x8 block as
// one contiguous run of 128-bit stores.
//
// K3 replaces src/models/network.py:172-262 (mask -> softmax -> Categorical sample/log_prob ->
// masked entropy): 8 lanes per row, 768 B of logits read once with 128-bit loads (128 B
// contiguous per row group per instruction), everything else in registers / 3-step butterflies.
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <math.h>
#include "bb_kernels.h"

__constant__ uint64_t c_piece_cells[BB_NUM_PIECES + 3] = BB_PIECE_MASKS;
__constant__ uint64_t c_piece_inb[BB_NUM_PIECES + 3] = BB_PIECE_INB;
__device__ const BBSymTables g_bb_sym = {BB_SYM_PERM, BB_SYM_SHIFT};

// ------------------------------------------------------------------------------------ K2
// One item = 16 output bytes, so consecutive lanes always store consecutive 16-byte pieces
// (full 32-byte sectors per instruction): bf16 item = (env, channel, row) -> 8 values,
// f32 item = (env, channel, row, half) -> 4 values.
// SYM (K7a): output row g*n + i is view g (bb_sym_board / BB_SYM_PERM, bb_rules.cuh) of input row i, so each
// view is a contiguous block of n rows; `perm` = the [8][40] piece permutation in shared memory.
template <bool BF16, bool SYM = false>
__device__ __forceinline__ uint64_t bb_obs_plane(const uint64_t* __restrict__ board, const uint32_t* __restrict__ pieces,
                                                 const uint64_t* cells, int64_t t, const int64_t* __restrict__ index = nullptr,
                                                 int64_t n = 0, const uint8_t* perm = nullptr) {
    int64_t env = t >> (BF16 ? 5 : 6);
    int g = 0;
    if (SYM) {
#pragma unroll
        for (int k = 1; k < BB_SYM_N; ++k) g += env >= k * n ? 1 : 0;
        env -= g * n;
    }
    if (index) env = __ldg(index + env);          // minibatch gather: output row -> rollout-buffer sample
    const int ch = (int)(t >> (BF16 ? 3 : 4)) & 3;
    if (ch == 0) return SYM ? bb_sym_board(g, __ldg(board + env)) : __ldg(board + env);
    const uint32_t pw = __ldg(pieces + env);
    uint32_t id = (pw >> (8 * (ch - 1))) & 0xFFu;
    if (SYM && id < BB_NUM_PIECES) id = perm[g * BB_TABLE_N + id];
    const bool used = (pw >> (24 + ch - 1)) & 1u;
    return used ? 0ull : cells[id < BB_NUM_PIECES ? id : BB_NUM_PIECES];
}

// split != NULL (f32 only): the reference's separate arrays — board planes f32[n][8][8] at `obs`, piece
// planes f32[n][3][8][8] at `split` (engine.get_observation, engine.py:489-507) — instead of one
// [n][4][8][8] block
template <bool BF16>
__device__ __forceinline__ void bb_unpack_obs_item(void* __restrict__ obs, int64_t t, uint64_t plane_bits,
                                                   void* __restrict__ split = nullptr) {
    if (!BF16 && split) {
        const int64_t env = t >> 6;
        const int ch = (int)(t >> 4) & 3, q = (int)t & 15;
        const uint32_t bits = (uint32_t)(plane_bits >> (4 * q)) & 0xFu;
        float4 v;
        v.x = (bits & 1u) ? 1.f : 0.f; v.y = (bits & 2u) ? 1.f : 0.f;
        v.z = (bits & 4u) ? 1.f : 0.f; v.w = (bits & 8u) ? 1.f : 0.f;
        if (ch == 0) __stcs(reinterpret_cast<float4*>(obs) + env * 16 + q, v);
        else __stcs(reinterpret_cast<float4*>(split) + env * 48 + (ch - 1) * 16 + q, v);
        return;
    }
    if (BF16) {
        const uint32_t bits = (uint32_t)(plane_bits >> (8 * ((int)t & 7))) & 0xFFu;
        uint32_t w[4];                              // bf16 1.0 = 0x3F80
#pragma unroll
        for (int k = 0; k < 4; ++k)
            w[k] = (((bits >> (2 * k)) & 1u) ? 0x3F80u : 0u) | (((bits >> (2 * k + 1)) & 1u) ? 0x3F800000u : 0u);
        __stcs(reinterpret_cast<uint4*>(obs) + t, make_uint4(w[0], w[1], w[2], w[3]));   // streaming: written once
    } else {
        const uint32_t bits = (uint32_t)(plane_bits >> (4 * ((int)t & 15))) & 0xFu;   // row*8 + half*4
        float4 v;
        v.x = (bits & 1u) ? 1.f : 0.f; v.y = (bits & 2u) ? 1.f : 0.f;
        v.z = (bits & 4u) ? 1.f : 0.f; v.w = (bits & 8u) ? 1.f : 0.f;
        __stcs(reinterpret_cast<float4*>(obs) + t, v);
    }
}

// Grid-stride: a few thousand long-lived blocks instead of one short block per 8 envs (CTA
// launch rate, not HBM, bounded the one-shot version); two independent items per iteration.
// SYM: the eight-view kernel K7a, 8n output rows (see bb_obs_plane).
template <bool BF16, bool SYM = false>
__global__ void __launch_bounds__(256)
bb_unpack_obs_kernel(const uint64_t* __restrict__ board, const uint32_t* __restrict__ pieces,
                     void* __restrict__ obs, int64_t n, void* __restrict__ split, const int64_t* __restrict__ index) {
    __shared__ uint64_t cells[BB_NUM_PIECES + 3];
    __shared__ uint8_t perm[SYM ? BB_SYM_N * BB_TABLE_N : 1];
    for (int k = threadIdx.x; k < BB_NUM_PIECES + 3; k += blockDim.x) cells[k] = c_piece_cells[k];
    if (SYM)
        for (int k = threadIdx.x; k < BB_SYM_N * BB_TABLE_N; k += blockDim.x) perm[k] = g_bb_sym.perm[k / BB_TABLE_N][k % BB_TABLE_N];
    __syncthreads();
    if (SYM) split = nullptr;
    const int64_t total = (SYM ? BB_SYM_N * n : n) * (BF16 ? 32 : 64);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    // SYM: one item per iteration (the four-item body spills with the view transforms inlined four times)
    for (; !SYM && t + 3 * stride < total; t += 4 * stride) {
        const uint64_t p0 = bb_obs_plane<BF16, SYM>(board, pieces, cells, t, index, n, perm);
        const uint64_t p1 = bb_obs_plane<BF16, SYM>(board, pieces, cells, t + stride, index, n, perm);
        const uint64_t p2 = bb_obs_plane<BF16, SYM>(board, pieces, cells, t + 2 * stride, index, n, perm);
        const uint64_t p3 = bb_obs_plane<BF16, SYM>(board, pieces, cells, t + 3 * stride, index, n, perm);
        bb_unpack_obs_item<BF16>(obs, t, p0, split);
        bb_unpack_obs_item<BF16>(obs, t + stride, p1, split);
        bb_unpack_obs_item<BF16>(obs, t + 2 * stride, p2, split);
        bb_unpack_obs_item<BF16>(obs, t + 3 * stride, p3, split);
    }
    for (; t < total; t += stride)
        bb_unpack_obs_item<BF16>(obs, t, bb_obs_plane<BF16, SYM>(board, pieces, cells, t, index, n, perm), split);
}

template <bool F32>
__global__ void __launch_bounds__(256)
bb_unpack_mask_kernel(const uint64_t* __restrict__ mask, int64_t stride, void* __restrict__ dense, int64_t n) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // (env, group of 16 actions)
    const int64_t env = t / 12;
    if (env >= n) return;
    const int g = (int)(t - env * 12);
    const uint64_t w = __ldg(mask + (int64_t)(g >> 2) * stride + env);
    const uint32_t bits = (uint32_t)(w >> (16 * (g & 3))) & 0xFFFFu;
    if (F32) {
        float4* o = reinterpret_cast<float4*>(dense) + 4 * t;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float4 v;
            v.x = ((bits >> (4 * k)) & 1u) ? 1.f : 0.f;
            v.y = ((bits >> (4 * k + 1)) & 1u) ? 1.f : 0.f;
            v.z = ((bits >> (4 * k + 2)) & 1u) ? 1.f : 0.f;
            v.w = ((bits >> (4 * k + 3)) & 1u) ? 1.f : 0.f;
            o[k] = v;
        }
    } else {
        uint32_t w4[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t nib = (bits >> (4 * k)) & 0xFu;
            w4[k] = (nib & 1u) | ((nib & 2u) << 7) | ((nib & 4u) << 14) | ((nib & 8u) << 21);
        }
        reinterpret_cast<uint4*>(dense)[t] = make_uint4(w4[0], w4[1], w4[2], w4[3]);
    }
}

static void bb_launch_obs_planes(const uint64_t* board, const uint32_t* pieces, void* obs, int obs_dtype, int64_t n,
                                 void* split, const int64_t* index, cudaStream_t stream, bool sym = false) {
    const int64_t threads = (sym ? BB_SYM_N * n : n) * (obs_dtype == 1 ? 32 : 64);
    int64_t blocks = (threads + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;        // grid-stride: 8 resident blocks per SM x 2 waves
    const unsigned grid = (unsigned)blocks;
    if (sym) {
        if (obs_dtype == 1) bb_unpack_obs_kernel<true, true><<<grid, 256, 0, stream>>>(board, pieces, obs, n, nullptr, index);
        else bb_unpack_obs_kernel<false, true><<<grid, 256, 0, stream>>>(board, pieces, obs, n, nullptr, index);
        return;
    }
    if (obs_dtype == 1) bb_unpack_obs_kernel<true><<<grid, 256, 0, stream>>>(board, pieces, obs, n, nullptr, index);
    else bb_unpack_obs_kernel<false><<<grid, 256, 0, stream>>>(board, pieces, obs, n, split, index);
}

cudaError_t bb_launch_unpack_obs_sym(const uint64_t* board, const uint32_t* pieces, const int64_t* index, void* obs,
                                     int obs_dtype, int64_t n, cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    bb_launch_obs_planes(board, pieces, obs, obs_dtype, n, nullptr, index, stream, true);
    return cudaGetLastError();
}

cudaError_t bb_launch_unpack_obs(const uint64_t* board, const uint32_t* pieces, const uint64_t* mask,
                                 int64_t mask_stride, void* obs_nchw, int obs_dtype, void* mask_dense,
                                 int mask_dtype, int64_t n, cudaStream_t stream, void* pieces_split) {
    if (n <= 0) return cudaSuccess;
    if (obs_nchw) bb_launch_obs_planes(board, pieces, obs_nchw, obs_dtype, n, pieces_split, nullptr, stream);
    if (mask_dense) {
        const int64_t threads = n * 12;
        const unsigned grid = (unsigned)((threads + 255) / 256);
        if (mask_dtype == 0) bb_unpack_mask_kernel<true><<<grid, 256, 0, stream>>>(mask, mask_stride, mask_dense, n);
        else bb_unpack_mask_kernel<false><<<grid, 256, 0, stream>>>(mask, mask_stride, mask_dense, n);
    }
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------ minibatch gather
// RolloutBuffer.get_samples (src/agents/ppo.py:171-213): the reference gathers seven arrays of
// 1.8 KB rows with numpy fancy indexing and uploads them.  Here sample index[b] of the packed
// device-resident buffer (board u64, pieces u32, mask planes [T][3][N], action, log-prob,
// advantage, return; T*N samples, flat index t*N + e) becomes row b of the minibatch: the obs
// planes are expanded by the K2 kernel reading through the index, the scalars and the mask planes
// [3][B] by one thread per row; advantages are normalised on the way, (a - mean) / (std + 1e-8) in
// float32 like ppo.py:196.
__global__ void __launch_bounds__(256)
bb_gather_rows_kernel(const int64_t* __restrict__ index, int64_t B, int64_t N, const uint64_t* __restrict__ mask,
                      const int32_t* __restrict__ action, const float* __restrict__ logp, const float* __restrict__ adv,
                      const float* __restrict__ ret, const float* __restrict__ mean_std, uint64_t* __restrict__ mask_out,
                      int32_t* __restrict__ action_out, float* __restrict__ logp_out, float* __restrict__ adv_out,
                      float* __restrict__ ret_out) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const int64_t j = index[b];
    const int64_t t = j / N, e = j - t * N;
    const uint64_t* m = mask + t * 3 * N + e;
    mask_out[b] = m[0]; mask_out[B + b] = m[N]; mask_out[2 * B + b] = m[2 * N];
    action_out[b] = action[j];
    logp_out[b] = logp[j];
    ret_out[b] = ret[j];
    const float a = adv[j];
    adv_out[b] = mean_std ? __fdiv_rn(__fsub_rn(a, mean_std[0]), __fadd_rn(mean_std[1], 1e-8f)) : a;
}

cudaError_t bb_launch_gather_minibatch(const int64_t* index, int64_t B, int64_t N, const uint64_t* board,
                                       const uint32_t* pieces, const uint64_t* mask, const int32_t* action,
                                       const float* logp, const float* adv, const float* ret, const float* mean_std,
                                       void* obs, int obs_dtype, uint64_t* mask_out, int32_t* action_out, float* logp_out,
                                       float* adv_out, float* ret_out, cudaStream_t stream) {
    if (B <= 0) return cudaSuccess;
    if (obs) bb_launch_obs_planes(board, pieces, obs, obs_dtype, B, nullptr, index, stream);
    bb_gather_rows_kernel<<<(unsigned)((B + 255) / 256), 256, 0, stream>>>(index, B, N, mask, action, logp, adv, ret, mean_std,
                                                                          mask_out, action_out, logp_out, adv_out, ret_out);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------ K3
// Backward / loss kernels: 8 lanes per row, 4 rows per warp; lane l of a row group owns the 24 actions
//     a(l,k,c) = 32k + 4l + c        k = 0..5, c = 0..3      (register index i = 4k + c)
// i.e. the k-th 128-bit load of the group is one contiguous 128 B (f32) run.  The forward kernel uses 4 lanes
// per row (see below).  Everything else is per-lane arithmetic plus butterflies inside the group.
// Maths (network.py:172-262):
//   e_i = 2^((z_i - m) log2 e)        one FFMA + one MUFU per action; masked actions carry z = -1e30,
//                                     so e_i is exactly 0 and every product with it stays finite
//   S = sum e_i,  log p_a = (z_a - m) - log S, clamped to [log eps, log(1 - eps)]   (torch Categorical
//                                     clamps the normalised probability, network.py:213-225)
//   entropy  = log S - sum_i e_i (z_i - m) / S   == -sum q log q (network.py:246-260); the reference's
//              clamps at 1e-10 change it by < 1e-8
// Sampling is the inverse CDF of u * S over the UNNORMALISED e_i in the order (lane, k, c) — a fixed
// permutation of the actions, so the draw is an exact categorical sample; philox.py documents the
// order.  The lane's running sums are its local CDF; the pick is the number of entries <= the
// threshold.  z_a of the chosen / given action is re-read from global memory (an L1 hit) instead of
// being selected out of 24 registers.  The first version of this layout normalised all 24
// probabilities, summed them again and selected p_a with 24 predicated moves per lane: ~700
// instructions per lane, instruction-bound at the same 103 us for f32 and bf16 logits; this one
// executes ~300.
#define K3_LOG2E 1.4426950408889634f
#define K3_LN2 0.6931471805599453f
#define K3_MASKED (-1.0e30f)   // stands in for -inf: 2^(K3_MASKED * log2e) == 0 and 0 * K3_MASKED == 0
#define K3_LOG_EPS (-15.942385152878742f)          // log(torch.finfo(float32).eps)
#define K3_LOG_1M_EPS (-1.1920929665620860e-07f)   // log(1 - eps)

__device__ __forceinline__ float k3_ex2(float x) {      // 2^x, one MUFU (rel. error 2^-22)
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__device__ __forceinline__ float grp_max(float v) {
    v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
    v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
    return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 4));
}
__device__ __forceinline__ float grp_sum(float v) {
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    return v + __shfl_xor_sync(0xffffffffu, v, 4);
}

// mask bits of this lane's 24 actions: bit (4k + c) = action 32k + 4l + c
__device__ __forceinline__ uint32_t k3_lane_mask(const uint64_t* __restrict__ mask, int64_t stride, int64_t row, int l) {
    uint32_t mb = 0;
#pragma unroll
    for (int p = 0; p < 3; ++p) {
        const uint64_t w = __ldg(mask + (int64_t)p * stride + row);
        mb |= ((uint32_t)(w >> (4 * l)) & 0xFu) << (8 * p);
        mb |= ((uint32_t)(w >> (32 + 4 * l)) & 0xFu) << (8 * p + 4);
    }
    return mb;
}

// this lane's 24 logits, masked ones replaced by K3_MASKED
template <bool BF16>
__device__ __forceinline__ void k3_load_row(const void* __restrict__ logits, int64_t row, int l, uint32_t mb, float z[24]) {
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        float4 v;
        if (BF16) {
            const uint2 h = reinterpret_cast<const uint2*>(logits)[row * 48 + k * 8 + l];
            v.x = __uint_as_float(h.x << 16); v.y = __uint_as_float(h.x & 0xFFFF0000u);
            v.z = __uint_as_float(h.y << 16); v.w = __uint_as_float(h.y & 0xFFFF0000u);
        } else {
            v = reinterpret_cast<const float4*>(logits)[row * 48 + k * 8 + l];
        }
        z[4 * k + 0] = v.x; z[4 * k + 1] = v.y; z[4 * k + 2] = v.z; z[4 * k + 3] = v.w;
    }
#pragma unroll
    for (int i = 0; i < 24; ++i) z[i] = ((mb >> i) & 1u) ? z[i] : K3_MASKED;      // masking (network.py:175-180)
}

template <bool BF16>
__device__ __forceinline__ float k3_logit(const void* __restrict__ logits, int64_t row, int a) {
    if (BF16) return __uint_as_float((uint32_t)reinterpret_cast<const uint16_t*>(logits)[row * 192 + a] << 16);
    return reinterpret_cast<const float*>(logits)[row * 192 + a];
}

// is action a (0..191) set in the three mask planes of `row`
__device__ __forceinline__ bool k3_action_valid(const uint64_t* __restrict__ mask, int64_t stride, int64_t row, int a) {
    if (a < 0 || a >= 192) return false;
    return (__ldg(mask + (int64_t)(a >> 6) * stride + row) >> (a & 63)) & 1ull;
}

// ---- forward: 4 lanes per row, 8 rows per warp.  Lane l of a row group owns the 48 actions
//     a(l,k,c) = 16k + 4l + c        k = 0..11, c = 0..3     (register index i = 4k + c)
// (the k-th load of the group is one contiguous 64 B (f32) / 32 B (bf16) run).  With 8 lanes per row the
// per-lane fixed work (Philox, mask unpack, prefix scan, logs: ~270 instructions) was paid eight times per
// row and outweighed the 24 x ~10 instructions of per-action arithmetic; four lanes halve that share.
// Warps walk the rows grid-stride, and one Philox evaluation per lane serves FOUR trips: lane 4g + i draws
// the uniform of row group g for trip j + i, the group picks it up with a shuffle (same stream position as
// before: keyed by seed, global row id and call counter only).
__device__ __forceinline__ float grp4_max(float v) {
    v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
    return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}
__device__ __forceinline__ float grp4_sum(float v) {
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    return v + __shfl_xor_sync(0xffffffffu, v, 2);
}

// mask bits of this lane's 48 actions: bit (4k + c) = action 16k + 4l + c; plane p holds k = 4p .. 4p+3
__device__ __forceinline__ uint64_t k3_lane_mask4(const uint64_t* __restrict__ mask, int64_t stride, int64_t row, int l) {
    uint64_t mb = 0;
#pragma unroll
    for (int p = 0; p < 3; ++p) {
        const uint64_t w = __ldg(mask + (int64_t)p * stride + row) >> (4 * l);
        const uint32_t lo = (uint32_t)w, hi = (uint32_t)(w >> 32);
        // nibbles at bits 0 and 16 of each half -> one byte per half
        const uint32_t b = (lo & 0xFu) | ((lo >> 12) & 0xF0u) | ((hi & 0xFu) << 8) | ((hi >> 4) & 0xF000u);
        mb |= (uint64_t)b << (16 * p);
    }
    return mb;
}

// MODE 0 sample, 1 argmax, 2 evaluate the given actions; ENT: also write the masked entropy.
// bf16 logits: 6 blocks per SM (80 registers) — the kernel is bound by the half-rate ALU pipe (select, max,
// compare, count, bf16 unpack: ~4 of the ~10 instructions per action) and by latency at 5 warps per
// scheduler; measured (tools/time_k3.py, sustained clocks) bf16 + entropy 83.5 -> 70.9 us with the bound,
// f32 85.6 -> 92.8 us, so f32 stays at 5 blocks (96 registers).
template <bool BF16, int MODE, bool ENT>
__global__ void __launch_bounds__(128, BF16 ? 6 : 5)
bb_masked_sample_kernel(const void* __restrict__ logits, const uint64_t* __restrict__ mask, int64_t stride,
                        uint64_t seed, uint64_t call_counter, int32_t* __restrict__ action,
                        float* __restrict__ logp_out, float* __restrict__ ent_out, int64_t n, int64_t row_offset,
                        const uint64_t* __restrict__ counter_dev) {
    const int lane = threadIdx.x & 31;
    const int l = lane & 3;                       // lane inside the row group
    const int g = lane >> 2;                      // row group of the warp
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const uint64_t ctr = MODE == 0 ? call_counter + (counter_dev ? *counter_dev : 0ull) : 0ull;
    uint32_t ubatch = 0;                          // Philox word of (group g, trip j - (j & 3) + l)
    int trip = 0;
    for (int64_t r0 = warp0 * 8; r0 < n; r0 += n_warps * 8, ++trip) {
    const int64_t row_raw = r0 + g;
    const bool live = row_raw < n;
    const int64_t row = live ? row_raw : n - 1;   // out-of-range groups shadow the last row, never store
    if (MODE == 0 && (trip & 3) == 0) {
        // keyed by the GLOBAL row id (env shards on several GPUs draw independent noise) and by a call
        // counter that may live on the device (a CUDA graph replays the launch with a new value)
        const uint64_t grow = (uint64_t)(r0 + (int64_t)l * n_warps * 8 + g + row_offset);
        ubatch = bb_philox((uint32_t)grow, (uint32_t)(grow >> 32), (uint32_t)ctr, BB_STREAM_SAMPLE,
                           (uint32_t)seed, (uint32_t)(seed >> 32)).x;
    }

    float z[48];
    const uint64_t mb = k3_lane_mask4(mask, stride, row, l);
#pragma unroll
    for (int k = 0; k < 12; ++k) {
        float4 v;
        if (BF16) {
            const uint2 h = reinterpret_cast<const uint2*>(logits)[row * 48 + k * 4 + l];
            v.x = __uint_as_float(h.x << 16); v.y = __uint_as_float(h.x & 0xFFFF0000u);
            v.z = __uint_as_float(h.y << 16); v.w = __uint_as_float(h.y & 0xFFFF0000u);
        } else {
            v = reinterpret_cast<const float4*>(logits)[row * 48 + k * 4 + l];
        }
        z[4 * k + 0] = v.x; z[4 * k + 1] = v.y; z[4 * k + 2] = v.z; z[4 * k + 3] = v.w;
    }
    const uint32_t mlo = (uint32_t)mb, mhi = (uint32_t)(mb >> 32);
    float m = K3_MASKED;
#pragma unroll
    for (int i = 0; i < 48; ++i) {
        const bool ok = i < 32 ? ((mlo >> i) & 1u) : ((mhi >> (i - 32)) & 1u);
        z[i] = ok ? z[i] : K3_MASKED;             // masking (network.py:175-180)
        m = fmaxf(m, z[i]);
    }
    m = grp4_max(m);
    const bool any_valid = m > 0.5f * K3_MASKED;
    const float nm2 = any_valid ? -m * K3_LOG2E : 0.f;
    // z[i] becomes the lane's running sum of e (its local CDF); sz2 = sum e_i d_i log2e
    float run = 0.f, sz2 = 0.f, best = K3_MASKED;
    int bi = 0;
#pragma unroll
    for (int i = 0; i < 48; ++i) {
        // argmax on the masked logit, not on e: two logits a few ulps apart can give equal e (or e in the
        // wrong order, ex2.approx is accurate to 2^-22 only)
        if (MODE == 1) { if (z[i] > best) { best = z[i]; bi = i; } }   // first maximum = lowest action index of the lane
        const float d2 = fmaf(z[i], K3_LOG2E, nm2);               // (z - m) log2e <= 0
        const float e = k3_ex2(d2);                               // exactly 0 for masked actions
        if (ENT) sz2 = fmaf(e, d2, sz2);
        run += e;
        z[i] = run;
    }
    const float lane_tot = run;
    const float s = grp4_sum(lane_tot);

    int act = 0;
    if (MODE == 2) {
        act = action[row];
    } else if (MODE == 1) {
        // argmax of the masked logits (= of probs), lowest action index on ties (torch.argmax)
        int idx = 16 * (bi >> 2) + 4 * l + (bi & 3);
#pragma unroll
        for (int d = 1; d < 4; d <<= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best, d);
            const int oi = __shfl_xor_sync(0xffffffffu, idx, d);
            if (ob > best || (ob == best && oi < idx)) { best = ob; idx = oi; }
        }
        act = any_valid ? idx : 0;
    } else {
        const uint32_t word = __shfl_sync(0xffffffffu, ubatch, trip & 3, 4);      // this trip's draw of the group
        const float u = (float)(word >> 8) * (1.0f / 16777216.0f);
        const float t = u * s;
        // inclusive prefix of the lane totals inside the group
        float incl = lane_tot;
#pragma unroll
        for (int d = 1; d < 4; d <<= 1) {
            const float o = __shfl_up_sync(0xffffffffu, incl, d, 4);
            if (l >= d) incl += o;
        }
        // first lane whose inclusive prefix exceeds t (and that has any probability mass)
        const unsigned hit = (__ballot_sync(0xffffffffu, incl > t && lane_tot > 0.f) >> (lane & 28)) & 0xFu;
        const unsigned nz = (__ballot_sync(0xffffffffu, lane_tot > 0.f) >> (lane & 28)) & 0xFu;
        // rounding can leave t >= total: fall back to the last lane with mass
        const int L = hit ? (__ffs((int)hit) - 1) : (nz ? (31 - __clz((int)nz)) : 0);
        // inside the lane: the pick is the number of CDF entries <= the local threshold (masked entries
        // repeat the previous value, so they are skipped together with it), at most its last valid one.
        // incl - lane_tot is the lane's exclusive prefix as a difference of rounded float sums: it can exceed
        // the true prefix (small mass in a lower lane, a + b rounded up), and a t in that gap would give a
        // negative threshold, cnt = 0 and the lane's first action whether or not it is valid.  With tl >= 0
        // the first entry whose CDF exceeds tl has e > 0, and masked entries have e == 0 exactly.
        const float tl = fmaxf(t - (incl - lane_tot), 0.f);
        int cnt = 0;
#pragma unroll
        for (int i = 0; i < 48; ++i) cnt += (z[i] <= tl) ? 1 : 0;
        const int last = 63 - __clzll((long long)(mb | 1ull));
        const int pick = cnt < last ? cnt : last;
        const int idx = 16 * (pick >> 2) + 4 * l + (pick & 3);
        act = __shfl_sync(0xffffffffu, idx, L, 4);
        if (!any_valid) act = 0;
    }
    const float szt = ENT ? grp4_sum(sz2) : 0.f;      // group reduction: executed by all lanes
    if (live && l == 0) {
        if (MODE != 2) action[row] = act;
        const float logS = any_valid ? logf(s) : 0.f;
        if (logp_out) {
            float lp = K3_LOG_1M_EPS;             // all-masked row: p = 1 clamped (the reference would produce NaN)
            if (any_valid) {
                const bool ok = MODE != 2 || k3_action_valid(mask, stride, row, act);
                const int a = ok ? act : 0;
                lp = ok ? fmaf(k3_logit<BF16>(logits, row, a), K3_LOG2E, nm2) * K3_LN2 - logS : K3_LOG_EPS;
                lp = fminf(fmaxf(lp, K3_LOG_EPS), K3_LOG_1M_EPS);
            }
            logp_out[row] = lp;
        }
        if (ENT && ent_out) ent_out[row] = any_valid ? (logS - szt * K3_LN2 / s) : 0.f;
    }
    }   // rows of this warp
}

// one resident wave at most (persistent warps walk the rows): blocks per SM from the occupancy calculator
template <typename K>
static unsigned k3_wave(K kernel) {
    int dev = 0, sms = 0, per_sm = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 128, 0);
    return (unsigned)((sms > 0 ? sms : 148) * (per_sm > 0 ? per_sm : 4));
}

template <bool BF16, int MODE>
static void k3_launch(bool ent, int64_t want, cudaStream_t stream, const void* logits, const uint64_t* mask, int64_t stride,
                      uint64_t seed, uint64_t call_counter, int32_t* action, float* logp, float* entropy, int64_t n,
                      int64_t row_offset, const uint64_t* counter_dev) {
    if (ent) {
        static const unsigned wave = k3_wave(bb_masked_sample_kernel<BF16, MODE, true>);
        const unsigned grid = (unsigned)(want < (int64_t)wave ? want : wave);
        bb_masked_sample_kernel<BF16, MODE, true><<<grid, 128, 0, stream>>>(logits, mask, stride, seed, call_counter, action, logp, entropy, n, row_offset, counter_dev);
    } else {
        static const unsigned wave = k3_wave(bb_masked_sample_kernel<BF16, MODE, false>);
        const unsigned grid = (unsigned)(want < (int64_t)wave ? want : wave);
        bb_masked_sample_kernel<BF16, MODE, false><<<grid, 128, 0, stream>>>(logits, mask, stride, seed, call_counter, action, logp, entropy, n, row_offset, counter_dev);
    }
}

cudaError_t bb_launch_masked_sample(const void* logits, int logits_dtype, const uint64_t* mask,
                                    int64_t mask_stride, uint64_t seed, uint64_t call_counter, int mode,
                                    int32_t* action, float* logp, float* entropy, int64_t n, cudaStream_t stream,
                                    int64_t row_offset, const uint64_t* counter_dev) {
    if (n <= 0) return cudaSuccess;
    const int64_t want = (n + 31) / 32;           // 32 rows per block and trip
    const bool ent = entropy != nullptr;
#define K3_GO(BF, MD) k3_launch<BF, MD>(ent, want, stream, logits, mask, mask_stride, seed, call_counter, action, logp, entropy, n, row_offset, counter_dev)
    if (logits_dtype == 1) {
        if (mode == 0) K3_GO(true, 0); else if (mode == 1) K3_GO(true, 1); else K3_GO(true, 2);
    } else {
        if (mode == 0) K3_GO(false, 0); else if (mode == 1) K3_GO(false, 1); else K3_GO(false, 2);
    }
#undef K3_GO
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------ K3 backward
// Gradient of (log_prob[action], masked entropy) w.r.t. the raw logits, for the PPO update
// (autograd of src/models/network.py:210-262 as used at src/agents/ppo.py:366-392):
//   d log_prob / d z_i = [eps <= p_a <= 1-eps] (delta_ia - p_i)        (Categorical clamps p)
//   d entropy  / d z_i = -p_i (log p_i + H)
// for valid actions i, 0 for masked ones.  Same 8-lanes-per-row layout as the forward; p is
// recomputed from the logits (768 B read + 768 B written per row, nothing saved between passes).
// With d_i = z_i - m, e_i = 2^(d_i log2e):
//   dlogits_i = e_i * (c0 + c1 d_i)      c1 = -g_ent / S,  c0 = (-g_logp - g_ent (H - log S)) / S
// i.e. FADD + FMUL + MUFU (e), FADD + FFMA (S and the entropy sum), FFMA + FMUL (gradient) per action; e_i is
// exactly 0 for masked actions, which zeroes their gradient without a select.  The delta term of the
// taken action is added by its owner lane with one scalar store after its vector stores (same thread,
// program order).
//
// LOSS = true turns the same pass into the whole PPO loss tail (src/agents/ppo.py:366-395 +
// network.py:210-262, SURVEY §8f item 2): with old log-probs, advantages, returns and the value
// head's output it forms ratio / clipped surrogate / value MSE / entropy bonus for the row,
// writes d(loss)/d(logits) and d(loss)/d(value) of
//     loss = mean(-min(r A, clip(r) A)) + value_coef mean((v - R)^2) - entropy_coef mean(H)
// directly (the loss is a mean with constant coefficients, so no second pass is needed), and adds
// the row's terms to five double sums: -min(..), (v-R)^2, H, (r-1) - log r, [|r-1| > clip].
struct BBPpoLossArgs {
    const float* old_logp; const float* adv; const float* ret; const float* value;
    float* dvalue; double* sums;
    float clip, value_coef, entropy_coef, inv_n;
};

template <bool BF16, bool LOSS>
__global__ void __launch_bounds__(128)
bb_masked_head_bwd_kernel(const void* __restrict__ logits, const uint64_t* __restrict__ mask, int64_t stride,
                          const int32_t* __restrict__ action, const float* __restrict__ g_logp,
                          const float* __restrict__ g_ent, void* __restrict__ dlogits, int64_t n, BBPpoLossArgs L) {
    const int lane = threadIdx.x & 31;
    const int l = lane & 7;
    // Warps walk the rows grid-stride, four rows per warp and trip (the loop bound is warp-uniform: the
    // shuffles below need all 32 lanes).  LOSS launches cap the grid (bb_launch_ppo_loss), so the five metric
    // sums leave each warp ONCE, after its last row: with one atomic set per four rows the 131,072 warps of
    // a 524,288-row call queued 655 k double atomics on five addresses and the kernel took 874 us, 15x its
    // memory time.
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f, t4 = 0.f;       // metric partial sums of this lane (LOSS)
    for (int64_t r0 = warp0 * 4; r0 < n; r0 += n_warps * 4) {
    const int64_t row_raw = r0 + (lane >> 3);
    const bool live = row_raw < n;
    const int64_t row = live ? row_raw : n - 1;
    float z[24], e[24];
    const uint32_t mb = k3_lane_mask(mask, stride, row, l);
    k3_load_row<BF16>(logits, row, l, mb, z);
    float m = K3_MASKED;
#pragma unroll
    for (int i = 0; i < 24; ++i) m = fmaxf(m, z[i]);
    m = grp_max(m);
    const bool any_valid = m > 0.5f * K3_MASKED;
    const float mm = any_valid ? m : 0.f;
    float s = 0.f, sz = 0.f;
#pragma unroll
    for (int i = 0; i < 24; ++i) {
        z[i] -= mm;                                // d = z - m: exactly 0 for the maximum (a one-action row gets an exactly zero gradient, like torch)
        e[i] = k3_ex2(z[i] * K3_LOG2E);            // exactly 0 where masked
        s += e[i];
        sz = fmaf(e[i], z[i], sz);
    }
    s = grp_sum(s);
    sz = grp_sum(sz);
    const float inv = any_valid ? __frcp_rn(s) : 0.f;
    const float logS = any_valid ? logf(s) : 0.f;
    const float H = logS - sz * inv;                // masked entropy
    const int act = action[row];
    const bool act_ok = any_valid && k3_action_valid(mask, stride, row, act);
    // z - m and p of the taken action (0 when it is masked / out of range)
    const float da = act_ok ? k3_logit<BF16>(logits, row, act) - mm : 0.f;
    const float pa = act_ok ? k3_ex2(da * K3_LOG2E) * inv : 0.f;
    const float eps = 1.1920928955078125e-07f;
    float g1, g2;
    if (LOSS) {
        const float logp = any_valid ? fminf(fmaxf(act_ok ? da - logS : K3_LOG_EPS, K3_LOG_EPS), K3_LOG_1M_EPS) : 0.f;
        const float lr = logp - L.old_logp[row];
        const float ratio = expf(lr);
        const float A = L.adv[row];
        const float s1 = ratio * A, s2 = fminf(fmaxf(ratio, 1.f - L.clip), 1.f + L.clip) * A;
        // d min(s1, s2) / d ratio: A where the unclipped term is the minimum (ties included: inside
        // the clip range both terms are the same function), 0 where the clipped constant is
        const bool through = s1 < s2 || (ratio >= 1.f - L.clip && ratio <= 1.f + L.clip);
        const float dv = L.value[row] - L.ret[row];
        g1 = (through && pa >= eps && pa <= 1.f - eps) ? -A * ratio * L.inv_n : 0.f;
        g2 = -L.entropy_coef * L.inv_n;
        // per-row metric terms: lane 0 of each 8-lane group accumulates them over the warp's rows
        if (live && l == 0) {
            L.dvalue[row] = 2.f * L.value_coef * dv * L.inv_n;
            t0 -= fminf(s1, s2); t1 = fmaf(dv, dv, t1); t2 += H; t3 += (ratio - 1.f) - lr;
            t4 += fabsf(ratio - 1.f) > L.clip ? 1.f : 0.f;
        }
    } else {
        g1 = (pa >= eps && pa <= 1.f - eps) ? g_logp[row] : 0.f;
        g2 = g_ent ? g_ent[row] : 0.f;
    }
    // dlogits_i = -g1 p_i - g2 p_i (log p_i + H),  log p_i = d_i - log S
    const float c1 = -g2 * inv;
    const float c0 = (-g1 - g2 * (H - logS)) * inv;
#pragma unroll
    for (int i = 0; i < 24; ++i) e[i] *= fmaf(z[i], c1, c0);
    if (live) {
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            if (BF16) {
                const __nv_bfloat162 a = __floats2bfloat162_rn(e[4 * k], e[4 * k + 1]);
                const __nv_bfloat162 b = __floats2bfloat162_rn(e[4 * k + 2], e[4 * k + 3]);
                uint2 h;
                h.x = *reinterpret_cast<const uint32_t*>(&a);
                h.y = *reinterpret_cast<const uint32_t*>(&b);
                reinterpret_cast<uint2*>(dlogits)[row * 48 + k * 8 + l] = h;
            } else {
                reinterpret_cast<float4*>(dlogits)[row * 48 + k * 8 + l] =
                    make_float4(e[4 * k], e[4 * k + 1], e[4 * k + 2], e[4 * k + 3]);
            }
        }
        // the delta term of the taken action, by the lane that owns (and has just stored) that element
        if (act_ok && g1 != 0.f && ((act & 31) >> 2) == l) {
            const float ga = k3_ex2(da * K3_LOG2E) * fmaf(da, c1, c0) + g1;
            if (BF16) reinterpret_cast<__nv_bfloat16*>(dlogits)[row * 192 + act] = __float2bfloat16_rn(ga);
            else reinterpret_cast<float*>(dlogits)[row * 192 + act] = ga;
        }
    }
    }   // rows of this warp
    if (LOSS) {
        // lanes 0, 8, 16, 24 hold the partial sums: fold them, one atomic per warp and sum
#pragma unroll
        for (int d = 8; d < 32; d <<= 1) {
            t0 += __shfl_xor_sync(0xffffffffu, t0, d); t1 += __shfl_xor_sync(0xffffffffu, t1, d);
            t2 += __shfl_xor_sync(0xffffffffu, t2, d); t3 += __shfl_xor_sync(0xffffffffu, t3, d);
            t4 += __shfl_xor_sync(0xffffffffu, t4, d);
        }
        if (lane == 0) {
            atomicAdd(&L.sums[0], (double)t0); atomicAdd(&L.sums[1], (double)t1); atomicAdd(&L.sums[2], (double)t2);
            atomicAdd(&L.sums[3], (double)t3); atomicAdd(&L.sums[4], (double)t4);
        }
    }
}

cudaError_t bb_launch_masked_head_bwd(const void* logits, int dtype, const uint64_t* mask, int64_t mask_stride,
                                      const int32_t* action, const float* g_logp, const float* g_ent,
                                      void* dlogits, int64_t n, cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    const unsigned grid = (unsigned)((n * 8 + 127) / 128);
    const BBPpoLossArgs none = {};
    if (dtype == 1)
        bb_masked_head_bwd_kernel<true, false><<<grid, 128, 0, stream>>>(logits, mask, mask_stride, action, g_logp, g_ent, dlogits, n, none);
    else
        bb_masked_head_bwd_kernel<false, false><<<grid, 128, 0, stream>>>(logits, mask, mask_stride, action, g_logp, g_ent, dlogits, n, none);
    return cudaGetLastError();
}

cudaError_t bb_launch_ppo_loss(const void* logits, int dtype, const uint64_t* mask, int64_t mask_stride,
                               const int32_t* action, const float* old_logp, const float* adv, const float* ret,
                               const float* value, float clip, float value_coef, float entropy_coef,
                               void* dlogits, float* dvalue, double* sums, int64_t n, cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    // one wave of 5 blocks per SM at most: every warp then walks n / 11,840 row quads and issues its five
    // atomics once, after its last row (float partial sums over at most a few hundred rows per lane)
    const int64_t want = (n * 8 + 127) / 128;
    const unsigned grid = (unsigned)(want < 148 * 5 ? want : 148 * 5);
    const BBPpoLossArgs L = {old_logp, adv, ret, value, dvalue, sums, clip, value_coef, entropy_coef, 1.0f / (float)n};
    if (dtype == 1)
        bb_masked_head_bwd_kernel<true, true><<<grid, 128, 0, stream>>>(logits, mask, mask_stride, action, nullptr, nullptr, dlogits, n, L);
    else
        bb_masked_head_bwd_kernel<false, true><<<grid, 128, 0, stream>>>(logits, mask, mask_stride, action, nullptr, nullptr, dlogits, n, L);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------ K7b
// Group average of the policy logits over the eight views (K7a rows g*n + i):
//   out[i, s*64 + a] = 0.125 * sum_{g = 0..7} L[g*n + i, s*64 + sigma_{g,p_s}(a)]      (f32, fixed g order)
// for an in-bounds anchor a of the slot's piece p_s, 0 elsewhere and for an id >= 37 (positions that are always
// masked).  The backward pass is the transposed map: every view position receives at most one term,
// 0.125 * dout, and 0 elsewhere.  A block stages the 8 x BB_K7B_STATES view rows of its states in shared memory
// with coalesced 16-byte accesses and does the permuted accesses there.  Per state: 8 x 768 B (f32) or
// 8 x 384 B (bf16) of logits and 768 B of f32 averages.
#define BB_K7B_STATES 4
#define BB_K7B_THREADS 256

__device__ __forceinline__ void k7b_load_tables(uint8_t* shift, uint64_t* inb) {
    for (int k = threadIdx.x; k < BB_SYM_N * BB_TABLE_N; k += blockDim.x) shift[k] = g_bb_sym.shift[k / BB_TABLE_N][k % BB_TABLE_N];
    for (int k = threadIdx.x; k < BB_TABLE_N; k += blockDim.x) inb[k] = k < BB_NUM_PIECES ? c_piece_inb[k] : 0ull;
}

// the piece id of output j (= s*64 + a) of a state with pieces word pw, or -1 where the output is always 0
__device__ __forceinline__ int k7b_piece(const uint64_t* inb, uint32_t pw, int j) {
    const uint32_t id = (pw >> (8 * (j >> 6))) & 0xFFu;
    return id < BB_NUM_PIECES && ((inb[id] >> (j & 63)) & 1ull) ? (int)id : -1;
}
// position of output j in the row of view g: s*64 + sigma_{g,id}(a)
__device__ __forceinline__ int k7b_pos(const uint8_t* shift, int id, int j, int g) {
    return (j & ~63) + bb_sym_cell(g, j & 63) - (int)shift[g * BB_TABLE_N + id];
}

template <bool BF16>
__global__ void __launch_bounds__(BB_K7B_THREADS)
bb_sym_logits_mean_kernel(const void* __restrict__ logits, const uint32_t* __restrict__ pieces, float* __restrict__ out,
                          int64_t n) {
    __shared__ float4 tile[BB_SYM_N * BB_K7B_STATES * 48];            // [g][state][192] as f32
    __shared__ uint8_t shift[BB_SYM_N * BB_TABLE_N];
    __shared__ uint64_t inb[BB_TABLE_N];
    k7b_load_tables(shift, inb);
    const float* tf = reinterpret_cast<const float*>(tile);
    for (int64_t i0 = (int64_t)blockIdx.x * BB_K7B_STATES; i0 < n; i0 += (int64_t)gridDim.x * BB_K7B_STATES) {
        const int ns = (int)(n - i0 < BB_K7B_STATES ? n - i0 : BB_K7B_STATES);
        // view g of the block's states is one contiguous run of rows g*n + i0 .. + ns
        constexpr int PER_ROW = BF16 ? 24 : 48;                       // 16-byte units per row
        for (int u = threadIdx.x; u < BB_SYM_N * BB_K7B_STATES * PER_ROW; u += blockDim.x) {
            const int g = u / (BB_K7B_STATES * PER_ROW), rem = u - g * (BB_K7B_STATES * PER_ROW);
            const int st = rem / PER_ROW, q = rem - st * PER_ROW;
            if (st >= ns) continue;
            const int64_t row = (int64_t)g * n + i0 + st;
            float4* dst = tile + (g * BB_K7B_STATES + st) * 48;
            if (BF16) {
                const uint4 h = __ldcs(reinterpret_cast<const uint4*>(logits) + row * 24 + q);
                dst[2 * q] = make_float4(__uint_as_float(h.x << 16), __uint_as_float(h.x & 0xFFFF0000u),
                                         __uint_as_float(h.y << 16), __uint_as_float(h.y & 0xFFFF0000u));
                dst[2 * q + 1] = make_float4(__uint_as_float(h.z << 16), __uint_as_float(h.z & 0xFFFF0000u),
                                             __uint_as_float(h.w << 16), __uint_as_float(h.w & 0xFFFF0000u));
            } else {
                dst[q] = __ldcs(reinterpret_cast<const float4*>(logits) + row * 48 + q);
            }
        }
        __syncthreads();
        for (int v = threadIdx.x; v < ns * 192; v += blockDim.x) {
            const int st = v / 192, j = v - st * 192;
            const int id = k7b_piece(inb, __ldg(pieces + i0 + st), j);
            float sum = 0.f;
            if (id >= 0) {
#pragma unroll
                for (int g = 0; g < BB_SYM_N; ++g) sum += tf[(g * BB_K7B_STATES + st) * 192 + k7b_pos(shift, id, j, g)];
            }
            out[(i0 + st) * 192 + j] = 0.125f * sum;             // read by K3 / the loss tail next: keep in L2
        }
        __syncthreads();
    }
}

template <bool BF16>
__global__ void __launch_bounds__(BB_K7B_THREADS)
bb_sym_logits_mean_bwd_kernel(const float* __restrict__ dout, const uint32_t* __restrict__ pieces, void* __restrict__ dlogits,
                              int64_t n) {
    __shared__ float4 tile[BB_SYM_N * BB_K7B_STATES * 48];
    __shared__ uint8_t shift[BB_SYM_N * BB_TABLE_N];
    __shared__ uint64_t inb[BB_TABLE_N];
    k7b_load_tables(shift, inb);
    float* tf = reinterpret_cast<float*>(tile);
    for (int64_t i0 = (int64_t)blockIdx.x * BB_K7B_STATES; i0 < n; i0 += (int64_t)gridDim.x * BB_K7B_STATES) {
        const int ns = (int)(n - i0 < BB_K7B_STATES ? n - i0 : BB_K7B_STATES);
        for (int u = threadIdx.x; u < BB_SYM_N * BB_K7B_STATES * 48; u += blockDim.x) tile[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        __syncthreads();
        for (int v = threadIdx.x; v < ns * 192; v += blockDim.x) {
            const int st = v / 192, j = v - st * 192;
            const int id = k7b_piece(inb, __ldg(pieces + i0 + st), j);
            if (id < 0) continue;
            const float d = 0.125f * __ldcs(dout + (i0 + st) * 192 + j);
#pragma unroll
            for (int g = 0; g < BB_SYM_N; ++g) tf[(g * BB_K7B_STATES + st) * 192 + k7b_pos(shift, id, j, g)] = d;
        }
        __syncthreads();
        constexpr int PER_ROW = BF16 ? 24 : 48;
        for (int u = threadIdx.x; u < BB_SYM_N * BB_K7B_STATES * PER_ROW; u += blockDim.x) {
            const int g = u / (BB_K7B_STATES * PER_ROW), rem = u - g * (BB_K7B_STATES * PER_ROW);
            const int st = rem / PER_ROW, q = rem - st * PER_ROW;
            if (st >= ns) continue;
            const int64_t row = (int64_t)g * n + i0 + st;
            const float4* src = tile + (g * BB_K7B_STATES + st) * 48;
            if (BF16) {
                const float4 a = src[2 * q], b = src[2 * q + 1];
                const __nv_bfloat162 h0 = __floats2bfloat162_rn(a.x, a.y), h1 = __floats2bfloat162_rn(a.z, a.w);
                const __nv_bfloat162 h2 = __floats2bfloat162_rn(b.x, b.y), h3 = __floats2bfloat162_rn(b.z, b.w);
                uint4 w;
                w.x = *reinterpret_cast<const uint32_t*>(&h0); w.y = *reinterpret_cast<const uint32_t*>(&h1);
                w.z = *reinterpret_cast<const uint32_t*>(&h2); w.w = *reinterpret_cast<const uint32_t*>(&h3);
                __stcs(reinterpret_cast<uint4*>(dlogits) + row * 24 + q, w);
            } else {
                __stcs(reinterpret_cast<float4*>(dlogits) + row * 48 + q, src[q]);
            }
        }
        __syncthreads();
    }
}

static unsigned k7b_grid(int64_t n) {
    const int64_t want = (n + BB_K7B_STATES - 1) / BB_K7B_STATES;
    return (unsigned)(want < 148 * 8 ? want : 148 * 8);        // grid-stride: one wave of 8 blocks per SM
}

cudaError_t bb_launch_sym_logits_mean(const void* logits, int dtype, const uint32_t* pieces, float* out, int64_t n,
                                      cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    if (dtype == 1) bb_sym_logits_mean_kernel<true><<<k7b_grid(n), BB_K7B_THREADS, 0, stream>>>(logits, pieces, out, n);
    else bb_sym_logits_mean_kernel<false><<<k7b_grid(n), BB_K7B_THREADS, 0, stream>>>(logits, pieces, out, n);
    return cudaGetLastError();
}

cudaError_t bb_launch_sym_logits_mean_bwd(const float* dout, const uint32_t* pieces, void* dlogits, int dtype, int64_t n,
                                          cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    if (dtype == 1) bb_sym_logits_mean_bwd_kernel<true><<<k7b_grid(n), BB_K7B_THREADS, 0, stream>>>(dout, pieces, dlogits, n);
    else bb_sym_logits_mean_bwd_kernel<false><<<k7b_grid(n), BB_K7B_THREADS, 0, stream>>>(dout, pieces, dlogits, n);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------ K7c
// Canonical frame: the network runs once per state, on the canonical view c(s) (bb_sym_canonical,
// bb_rules.cuh), and its logits are mapped back into the state's own frame.  With M(s) the view set
// (bit g set iff view g of s is c(s)):
//   out[i, s*64 + a] = (1/|M|) * sum_{g in M, ascending} L[i, s*64 + sigma_{g,p_s}(a)]      (f32)
// for an in-bounds anchor a of the slot's piece p_s (< 37) of the state's OWN pieces word, 0 elsewhere: the
// positions and zeros of K7b, restricted to the views that equal c(s).  1/|M| is a power of two.
// bb_sym_canonical_kernel: one thread per state, 12 B read (+ 8 B of index), 13 B written; the canonical
// rows then go through the unchanged K2.
__global__ void __launch_bounds__(256)
bb_sym_canonical_kernel(const uint64_t* __restrict__ board, const uint32_t* __restrict__ pieces,
                        const int64_t* __restrict__ index, uint64_t* __restrict__ cboard, uint32_t* __restrict__ cpieces,
                        uint8_t* __restrict__ views, int64_t n) {
    __shared__ BBSymTables S;                                   // only perm is read (bb_sym_pieces)
    for (int k = threadIdx.x; k < BB_SYM_N * BB_TABLE_N; k += blockDim.x) S.perm[k / BB_TABLE_N][k % BB_TABLE_N] = g_bb_sym.perm[k / BB_TABLE_N][k % BB_TABLE_N];
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = index ? __ldg(index + i) : i;
        uint64_t cb;
        uint32_t cp;
        views[i] = (uint8_t)bb_sym_canonical(&S, __ldg(board + r), __ldg(pieces + r), &cb, &cp);
        cboard[i] = cb;
        cpieces[i] = cp;
    }
}

// K7b's 16-byte staging of a logit row (f32 or bf16 in HBM <-> f32 in shared memory).  The K7b kernels keep
// their inline copies, which compile to the same instructions as before this section was added.
template <bool BF16>
__device__ __forceinline__ void k7c_stage(const void* __restrict__ logits, int64_t row, int q, float4* dst) {
    if (BF16) {
        const uint4 h = __ldcs(reinterpret_cast<const uint4*>(logits) + row * 24 + q);
        dst[2 * q] = make_float4(__uint_as_float(h.x << 16), __uint_as_float(h.x & 0xFFFF0000u),
                                 __uint_as_float(h.y << 16), __uint_as_float(h.y & 0xFFFF0000u));
        dst[2 * q + 1] = make_float4(__uint_as_float(h.z << 16), __uint_as_float(h.z & 0xFFFF0000u),
                                     __uint_as_float(h.w << 16), __uint_as_float(h.w & 0xFFFF0000u));
    } else {
        dst[q] = __ldcs(reinterpret_cast<const float4*>(logits) + row * 48 + q);
    }
}
template <bool BF16>
__device__ __forceinline__ void k7c_unstage(void* __restrict__ dlogits, int64_t row, int q, const float4* src) {
    if (BF16) {
        const float4 a = src[2 * q], b = src[2 * q + 1];
        const __nv_bfloat162 h0 = __floats2bfloat162_rn(a.x, a.y), h1 = __floats2bfloat162_rn(a.z, a.w);
        const __nv_bfloat162 h2 = __floats2bfloat162_rn(b.x, b.y), h3 = __floats2bfloat162_rn(b.z, b.w);
        uint4 w;
        w.x = *reinterpret_cast<const uint32_t*>(&h0); w.y = *reinterpret_cast<const uint32_t*>(&h1);
        w.z = *reinterpret_cast<const uint32_t*>(&h2); w.w = *reinterpret_cast<const uint32_t*>(&h3);
        __stcs(reinterpret_cast<uint4*>(dlogits) + row * 24 + q, w);
    } else {
        __stcs(reinterpret_cast<float4*>(dlogits) + row * 48 + q, src[q]);
    }
}

// 1/|M| (exact: |M| is 1, 2, 4 or 8); an empty view set gives 0
__device__ __forceinline__ float k7c_scale(uint32_t views) {
    const int c = __popc(views);
    return c ? 1.f / (float)c : 0.f;
}

#define BB_K7C_STATES 16

// Forward: a block stages the logit rows of BB_K7C_STATES states (one row each, contiguous) and gathers
// from them.  Per state: 768 B (f32) or 384 B (bf16) of logits, 4 B pieces, 1 B views, 768 B of f32 out.
template <bool BF16>
__global__ void __launch_bounds__(BB_K7B_THREADS)
bb_sym_logits_canonical_kernel(const void* __restrict__ logits, const uint32_t* __restrict__ pieces,
                               const uint8_t* __restrict__ views, float* __restrict__ out, int64_t n) {
    __shared__ float4 tile[BB_K7C_STATES * 48];
    __shared__ uint8_t shift[BB_SYM_N * BB_TABLE_N];
    __shared__ uint64_t inb[BB_TABLE_N];
    k7b_load_tables(shift, inb);
    const float* tf = reinterpret_cast<const float*>(tile);
    constexpr int PER_ROW = BF16 ? 24 : 48;
    for (int64_t i0 = (int64_t)blockIdx.x * BB_K7C_STATES; i0 < n; i0 += (int64_t)gridDim.x * BB_K7C_STATES) {
        const int ns = (int)(n - i0 < BB_K7C_STATES ? n - i0 : BB_K7C_STATES);
        for (int u = threadIdx.x; u < ns * PER_ROW; u += blockDim.x) {
            const int st = u / PER_ROW;
            k7c_stage<BF16>(logits, i0 + st, u - st * PER_ROW, tile + st * 48);
        }
        __syncthreads();
        for (int v = threadIdx.x; v < ns * 192; v += blockDim.x) {
            const int st = v / 192, j = v - st * 192;
            const int id = k7b_piece(inb, __ldg(pieces + i0 + st), j);
            const uint32_t vm = __ldg(views + i0 + st);
            float sum = 0.f;
            if (id >= 0) {
#pragma unroll
                for (int g = 0; g < BB_SYM_N; ++g)
                    if ((vm >> g) & 1u) sum += tf[st * 192 + k7b_pos(shift, id, j, g)];
            }
            out[(i0 + st) * 192 + j] = k7c_scale(vm) * sum;    // read by K3 / the loss tail next: keep in L2
        }
        __syncthreads();
    }
}

// Backward: the transposed map as a gather, so that a canonical position that several (g, j) pairs reach
// (|M| > 1: a stabiliser element maps the state onto itself) sums its terms in ascending g, the same order
// in every run.  Position k = s*64 + b of the canonical row is reached from view g in M exactly when b is an
// in-bounds anchor of the canonical slot's piece q = PERM[g][p_s] (the same for every g in M), from
// a = T_{g^-1}(b + SHIFT[g][p_s]) (sigma_{g,p} is a bijection of in-bounds anchors); elsewhere it is 0.
template <bool BF16>
__global__ void __launch_bounds__(BB_K7B_THREADS)
bb_sym_logits_canonical_bwd_kernel(const float* __restrict__ dout, const uint32_t* __restrict__ pieces,
                                   const uint8_t* __restrict__ views, void* __restrict__ dlogits, int64_t n) {
    __shared__ float4 din[BB_K7C_STATES * 48];                  // grad_out rows
    __shared__ float4 dst[BB_K7C_STATES * 48];                  // grad_logits rows
    __shared__ uint8_t shift[BB_SYM_N * BB_TABLE_N];
    __shared__ uint8_t perm[BB_SYM_N * BB_TABLE_N];
    __shared__ uint64_t inb[BB_TABLE_N];
    k7b_load_tables(shift, inb);
    for (int k = threadIdx.x; k < BB_SYM_N * BB_TABLE_N; k += blockDim.x) perm[k] = g_bb_sym.perm[k / BB_TABLE_N][k % BB_TABLE_N];
    const float* fin = reinterpret_cast<const float*>(din);
    float* fdst = reinterpret_cast<float*>(dst);
    constexpr int PER_ROW = BF16 ? 24 : 48;
    for (int64_t i0 = (int64_t)blockIdx.x * BB_K7C_STATES; i0 < n; i0 += (int64_t)gridDim.x * BB_K7C_STATES) {
        const int ns = (int)(n - i0 < BB_K7C_STATES ? n - i0 : BB_K7C_STATES);
        for (int u = threadIdx.x; u < ns * 48; u += blockDim.x) din[u] = __ldcs(reinterpret_cast<const float4*>(dout) + i0 * 48 + u);
        __syncthreads();
        for (int v = threadIdx.x; v < ns * 192; v += blockDim.x) {
            const int st = v / 192, k = v - st * 192;
            const uint32_t pw = __ldg(pieces + i0 + st), vm = __ldg(views + i0 + st);
            const uint32_t p = (pw >> (8 * (k >> 6))) & 0xFFu;
            const int b = k & 63;
            float sum = 0.f;
            if (p < BB_NUM_PIECES && vm && ((inb[perm[(__ffs(vm) - 1) * BB_TABLE_N + p]] >> b) & 1ull)) {
#pragma unroll
                for (int g = 0; g < BB_SYM_N; ++g)
                    if ((vm >> g) & 1u)
                        sum += fin[st * 192 + (k & ~63) + bb_sym_cell(bb_sym_inverse(g), b + (int)shift[g * BB_TABLE_N + p])];
            }
            fdst[v] = k7c_scale(vm) * sum;
        }
        __syncthreads();
        for (int u = threadIdx.x; u < ns * PER_ROW; u += blockDim.x) {
            const int st = u / PER_ROW;
            k7c_unstage<BF16>(dlogits, i0 + st, u - st * PER_ROW, dst + st * 48);
        }
        __syncthreads();
    }
}

static unsigned k7c_grid(int64_t n, int per_block) {
    const int64_t want = (n + per_block - 1) / per_block;
    return (unsigned)(want < 148 * 8 ? want : 148 * 8);        // grid-stride: one wave of 8 blocks per SM
}

cudaError_t bb_launch_sym_canonical(const uint64_t* board, const uint32_t* pieces, const int64_t* index, uint64_t* cboard,
                                    uint32_t* cpieces, uint8_t* views, int64_t n, cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    const int64_t blocks = (n + 255) / 256;
    bb_sym_canonical_kernel<<<(unsigned)(blocks < 148 * 16 ? blocks : 148 * 16), 256, 0, stream>>>(board, pieces, index, cboard,
                                                                                                  cpieces, views, n);
    return cudaGetLastError();
}

cudaError_t bb_launch_sym_logits_canonical(const void* logits, int dtype, const uint32_t* pieces, const uint8_t* views,
                                           float* out, int64_t n, cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    const unsigned grid = k7c_grid(n, BB_K7C_STATES);
    if (dtype == 1) bb_sym_logits_canonical_kernel<true><<<grid, BB_K7B_THREADS, 0, stream>>>(logits, pieces, views, out, n);
    else bb_sym_logits_canonical_kernel<false><<<grid, BB_K7B_THREADS, 0, stream>>>(logits, pieces, views, out, n);
    return cudaGetLastError();
}

cudaError_t bb_launch_sym_logits_canonical_bwd(const float* dout, const uint32_t* pieces, const uint8_t* views, void* dlogits,
                                               int dtype, int64_t n, cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    const unsigned grid = k7c_grid(n, BB_K7C_STATES);
    if (dtype == 1) bb_sym_logits_canonical_bwd_kernel<true><<<grid, BB_K7B_THREADS, 0, stream>>>(dout, pieces, views, dlogits, n);
    else bb_sym_logits_canonical_bwd_kernel<false><<<grid, BB_K7B_THREADS, 0, stream>>>(dout, pieces, views, dlogits, n);
    return cudaGetLastError();
}
