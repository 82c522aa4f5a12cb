// bb_bn_kernels.cu — training-mode BatchNorm + ReLU (+ residual add) for the policy CNN's
// channels-last bf16 activations (reference src/models/network.py:14-31, 78-92: every conv of
// the encoder is followed by BatchNorm2d + ReLU, the second one of a residual block by
// BatchNorm2d, "+ x", ReLU).
//
// The convolutions stay cuDNN/PyTorch.  What is replaced is the memory-bound glue around them:
// in the PPO update torch spends 70 % of the CNN's time in seven BatchNorm layers and their
// ReLU / add kernels (batch_norm_collect_statistics_channels_last 0.99 ms per layer on a
// 32,768 x 128 x 8 x 8 bf16 tensor = 0.54 TB/s).  Here a layer is
//   forward : one read of x for the statistics, one read of x (+ skip) and one write of y
//   backward: one read of (x, y, dy) for the two reductions, one more for dx (+ dskip)
// with 16-byte accesses and fp32 accumulation, i.e. HBM-roofline passes over [M = N*H*W, C].
//
// Layout: x, y, dy, dx, skip, dskip are [M, C] bf16, C a multiple of 8 (channels-last NHWC
// memory); gamma/beta/running stats/saved mean/rstd/dgamma/dbeta are fp32 [C].
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "bb_kernels.h"

#define BN_THREADS 256

struct BF8 { float v[8]; };

__device__ __forceinline__ BF8 bn_unpack(const uint4 q) {
    BF8 r;
    r.v[0] = __uint_as_float(q.x << 16); r.v[1] = __uint_as_float(q.x & 0xFFFF0000u);
    r.v[2] = __uint_as_float(q.y << 16); r.v[3] = __uint_as_float(q.y & 0xFFFF0000u);
    r.v[4] = __uint_as_float(q.z << 16); r.v[5] = __uint_as_float(q.z & 0xFFFF0000u);
    r.v[6] = __uint_as_float(q.w << 16); r.v[7] = __uint_as_float(q.w & 0xFFFF0000u);
    return r;
}

// the affine pair of the forward pass, y = relu(x * scale + shift): ONE definition, because the backward pass of
// layers without a residual input recomputes the ReLU mask from x with it instead of reading y back
__device__ __forceinline__ float bn_scale(float gamma, float rstd) { return __fmul_rn(gamma, rstd); }
__device__ __forceinline__ float bn_shift(float beta, float mean, float scale) { return __fmaf_rn(-mean, scale, beta); }

__device__ __forceinline__ uint32_t bn_pack2(float a, float b) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&h);
}

__device__ __forceinline__ uint4 bn_pack(const BF8& r) {
    return make_uint4(bn_pack2(r.v[0], r.v[1]), bn_pack2(r.v[2], r.v[3]), bn_pack2(r.v[4], r.v[5]), bn_pack2(r.v[6], r.v[7]));
}

// Two per-channel sums over the rows.  Thread t owns channel group t % G (8 channels) and walks
// the rows t / G, t / G + R, ... of its block's share; the block folds its row lanes in shared
// memory and writes ONE partial per channel to part[block][2][C] (no atomics: the finalize
// kernel adds the partials in a fixed order, so results are bit-reproducible).
//   MODE 0: sum (x - K), sum (x - K)^2, K = x[row 0]        (forward statistics; shifted by a value of the
//           channel so that q/M - (s/M)^2 does not cancel: with K = 0 the fp32 rounding left in sum x^2,
//           ~u x^2, is of the order of eps for |x| >~ 3 and a constant channel got var ~ 3e-5 instead of 0)
//   MODE 1: sum g, sum g * xhat, g = dy * [y > 0]           (backward reductions)
//   MODE 2: the same with the ReLU mask recomputed from x, [x * scale + shift > 0] with the forward's own
//           scale / shift expressions — layers without a residual input do not need y read back at all
template <int MODE>
__global__ void __launch_bounds__(BN_THREADS)
bb_bn_reduce_kernel(const uint4* __restrict__ x, const uint4* __restrict__ y, const uint4* __restrict__ dy,
                    const float* __restrict__ mean, const float* __restrict__ rstd, float* __restrict__ part,
                    int64_t M, int C, const float* __restrict__ gamma = nullptr, const float* __restrict__ beta = nullptr) {
    extern __shared__ float sh[];                      // [R][2][C]
    const int G = C >> 3, R = BN_THREADS / G;
    const int g = threadIdx.x % G, r0 = threadIdx.x / G;
    float a[8], b[8], mu[8], rs[8], sc[8], sf[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) { a[k] = 0.f; b[k] = 0.f; mu[k] = 0.f; rs[k] = 1.f; }
    if (MODE == 0 && r0 < R) {                         // the shift K = row 0 (x - K is exact in fp32 for bf16
        const BF8 k0 = bn_unpack(__ldg(x + g));        // values within a factor 2^15 of each other in magnitude)
#pragma unroll
        for (int k = 0; k < 8; ++k) mu[k] = k0.v[k];
    }
    if (MODE >= 1) {
#pragma unroll
        for (int k = 0; k < 8; ++k) { mu[k] = mean[g * 8 + k]; rs[k] = rstd[g * 8 + k]; }
    }
    if (MODE == 2) {
#pragma unroll
        for (int k = 0; k < 8; ++k) { sc[k] = bn_scale(gamma[g * 8 + k], rs[k]); sf[k] = bn_shift(beta[g * 8 + k], mu[k], sc[k]); }
    }
    if (r0 < R) {
        // U rows in flight per thread (all loads issued before the arithmetic): one 16-byte load per row kept
        // the forward pass at 0.75 of the HBM peak.  The rows are still accumulated in the same order.
        constexpr int U = MODE == 0 ? 4 : 2;
        const int64_t stride = (int64_t)gridDim.x * R;
        for (int64_t row = (int64_t)blockIdx.x * R + r0; row < M; row += U * stride) {
            uint4 xq[U], yq[U], dq[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int64_t rr = row + u * stride;
                if (rr < M) {
                    xq[u] = __ldg(x + rr * G + g);
                    if (MODE == 1) yq[u] = __ldg(y + rr * G + g);
                    if (MODE >= 1) dq[u] = __ldg(dy + rr * G + g);
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (row + u * stride >= M) continue;
                const BF8 xv = bn_unpack(xq[u]);
                if (MODE == 0) {
#pragma unroll
                    for (int k = 0; k < 8; ++k) { const float d = xv.v[k] - mu[k]; a[k] += d; b[k] = fmaf(d, d, b[k]); }
                } else if (MODE == 1) {
                    const BF8 yv = bn_unpack(yq[u]);
                    const BF8 dv = bn_unpack(dq[u]);
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const float gk = yv.v[k] > 0.f ? dv.v[k] : 0.f;
                        a[k] += gk;
                        b[k] = fmaf(gk, (xv.v[k] - mu[k]) * rs[k], b[k]);
                    }
                } else {
                    const BF8 dv = bn_unpack(dq[u]);
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const float gk = fmaf(xv.v[k], sc[k], sf[k]) > 0.f ? dv.v[k] : 0.f;
                        a[k] += gk;
                        b[k] = fmaf(gk, (xv.v[k] - mu[k]) * rs[k], b[k]);
                    }
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) { sh[(r0 * 2 + 0) * C + g * 8 + k] = a[k]; sh[(r0 * 2 + 1) * C + g * 8 + k] = b[k]; }
    }
    __syncthreads();
    for (int c = threadIdx.x; c < 2 * C; c += BN_THREADS) {
        float s = 0.f;
        for (int r = 0; r < R; ++r) s += sh[r * 2 * C + c];
        part[(int64_t)blockIdx.x * 2 * C + c] = s;
    }
}

// one BLOCK per channel adds that channel's two partial sums over the reduce kernel's blocks: thread t takes
// partials t, t + 256, ... (a handful of independent loads each — with one warp per channel every lane walked
// 37 dependent L2 round trips, 12 us per layer, 9 % of a 2,048-sample PPO step), then a fixed-order tree in
// shared memory; double accumulation, bit-reproducible.  Valid in thread 0.
#define BN_FIN_THREADS 256
__device__ __forceinline__ void bn_sum_partials(const float* __restrict__ part, int nblocks, int C, int c, double& s, double& q) {
    __shared__ double sh_s[BN_FIN_THREADS], sh_q[BN_FIN_THREADS];
    const int t = threadIdx.x;
    s = 0.0; q = 0.0;
    for (int b = t; b < nblocks; b += BN_FIN_THREADS) { s += (double)part[(int64_t)b * 2 * C + c]; q += (double)part[(int64_t)b * 2 * C + C + c]; }
    sh_s[t] = s; sh_q[t] = q;
    __syncthreads();
#pragma unroll
    for (int d = BN_FIN_THREADS / 2; d > 0; d >>= 1) {
        if (t < d) { sh_s[t] += sh_s[t + d]; sh_q[t] += sh_q[t + d]; }
        __syncthreads();
    }
    s = sh_s[0]; q = sh_q[0];
}

// forward finalize: mean / rstd of the batch, running statistics (momentum update with the
// unbiased variance, as torch.nn.BatchNorm2d), and the affine pair y = x * scale + shift.
// The partials are shifted sums of x - K (K = x[row 0][c], see MODE 0): mu = K + s/M, var = q/M - (s/M)^2.
__global__ void bb_bn_finalize_fwd_kernel(const float* __restrict__ part, int nblocks, int64_t M, int C, float eps,
                                          float momentum, const float* __restrict__ gamma, const float* __restrict__ beta,
                                          const float* __restrict__ pre_bias, float* __restrict__ running_mean, float* __restrict__ running_var,
                                          float* __restrict__ save_mean, float* __restrict__ save_rstd,
                                          float* __restrict__ scale, float* __restrict__ shift, const __nv_bfloat16* __restrict__ x) {
    const int c = blockIdx.x;                     // one block per channel
    double s, q;
    bn_sum_partials(part, nblocks, C, c, s, q);
    if (threadIdx.x != 0) return;
    const double d = s / (double)M;
    const double mu = (double)__bfloat162float(x[c]) + d;
    double var = q / (double)M - d * d;
    var = var > 0.0 ? var : 0.0;
    const float rstd = (float)(1.0 / sqrt(var + (double)eps));
    save_mean[c] = (float)mu;
    save_rstd[c] = rstd;
    if (running_mean) {
        const double unbiased = M > 1 ? var * (double)M / (double)(M - 1) : var;
        // a per-channel bias the caller left out of x (the conv bias: BatchNorm cancels it in y)
        // still belongs to the mean the module tracks
        running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * ((float)mu + (pre_bias ? pre_bias[c] : 0.f));
        running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
    }
    const float sc = bn_scale(gamma[c], rstd);
    scale[c] = sc;
    shift[c] = bn_shift(beta[c], (float)mu, sc);
}

// eval mode: the affine pair from the running statistics
__global__ void bb_bn_affine_eval_kernel(const float* __restrict__ gamma, const float* __restrict__ beta,
                                         const float* __restrict__ pre_bias, const float* __restrict__ running_mean, const float* __restrict__ running_var,
                                         float eps, int C, float* __restrict__ scale, float* __restrict__ shift) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const float sc = gamma[c] * rsqrtf(running_var[c] + eps);
    scale[c] = sc;
    shift[c] = beta[c] + ((pre_bias ? pre_bias[c] : 0.f) - running_mean[c]) * sc;
}

// y = relu(x * scale + shift (+ skip)); four rows in flight per thread
__global__ void __launch_bounds__(BN_THREADS)
bb_bn_apply_kernel(const uint4* __restrict__ x, const uint4* __restrict__ skip, const float* __restrict__ scale,
                   const float* __restrict__ shift, uint4* __restrict__ y, int64_t M, int C) {
    const int G = C >> 3, R = BN_THREADS / G;
    const int g = threadIdx.x % G, r0 = threadIdx.x / G;
    if (r0 >= R) return;
    float sc[8], sf[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) { sc[k] = scale[g * 8 + k]; sf[k] = shift[g * 8 + k]; }
    const int64_t stride = (int64_t)gridDim.x * R;
    for (int64_t row = (int64_t)blockIdx.x * R + r0; row < M; row += 4 * stride) {
        uint4 xq[4], sq[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int64_t rr = row + u * stride;
            if (rr < M) {
                xq[u] = __ldg(x + rr * G + g);
                if (skip) sq[u] = __ldg(skip + rr * G + g);
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int64_t rr = row + u * stride;
            if (rr < M) {
                BF8 v = bn_unpack(xq[u]);
                if (skip) {
                    const BF8 s = bn_unpack(sq[u]);
#pragma unroll
                    for (int k = 0; k < 8; ++k) v.v[k] = fmaxf(fmaf(v.v[k], sc[k], sf[k]) + s.v[k], 0.f);
                } else {
#pragma unroll
                    for (int k = 0; k < 8; ++k) v.v[k] = fmaxf(fmaf(v.v[k], sc[k], sf[k]), 0.f);
                }
                y[rr * G + g] = bn_pack(v);
            }
        }
    }
}

// backward finalize: dgamma, dbeta and the per-channel coefficients of
//   dx = scale * (g - c1 - xhat * c2),  c1 = sum g / M,  c2 = sum g xhat / M
__global__ void bb_bn_finalize_bwd_kernel(const float* __restrict__ part, int nblocks, int64_t M, int C,
                                          float* __restrict__ dgamma, float* __restrict__ dbeta,
                                          float* __restrict__ c1, float* __restrict__ c2) {
    const int c = blockIdx.x;                     // one block per channel
    double s, q;
    bn_sum_partials(part, nblocks, C, c, s, q);
    if (threadIdx.x != 0) return;
    dbeta[c] = (float)s;
    dgamma[c] = (float)q;
    c1[c] = (float)(s / (double)M);
    c2[c] = (float)(q / (double)M);
}

template <bool NOY>      // NOY: ReLU mask recomputed from x (no residual input), y is not read
__global__ void __launch_bounds__(BN_THREADS)
bb_bn_dx_kernel(const uint4* __restrict__ x, const uint4* __restrict__ y, const uint4* __restrict__ dy,
                const float* __restrict__ mean, const float* __restrict__ rstd, const float* __restrict__ gamma,
                const float* __restrict__ c1, const float* __restrict__ c2, uint4* __restrict__ dx,
                uint4* __restrict__ dskip, int64_t M, int C, const float* __restrict__ beta = nullptr) {
    const int G = C >> 3, R = BN_THREADS / G;
    const int g = threadIdx.x % G, r0 = threadIdx.x / G;
    if (r0 >= R) return;
    float mu[8], rs[8], sc[8], k1[8], k2[8], sf[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int c = g * 8 + k;
        mu[k] = mean[c]; rs[k] = rstd[c]; sc[k] = bn_scale(gamma[c], rs[k]); k1[k] = c1[c]; k2[k] = c2[c];
        sf[k] = NOY ? bn_shift(beta[c], mu[k], sc[k]) : 0.f;
    }
    constexpr int U = NOY ? 3 : 2;               // rows in flight: six 16-byte loads per thread either way
    const int64_t stride = (int64_t)gridDim.x * R;
    for (int64_t row = (int64_t)blockIdx.x * R + r0; row < M; row += U * stride) {
        uint4 xq[U], yq[U], dq[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t rr = row + u * stride;
            if (rr < M) { xq[u] = __ldg(x + rr * G + g); if (!NOY) yq[u] = __ldg(y + rr * G + g); dq[u] = __ldg(dy + rr * G + g); }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t rr = row + u * stride;
            if (rr < M) {
                const BF8 xv = bn_unpack(xq[u]), dv = bn_unpack(dq[u]);
                BF8 yv;
                if (!NOY) yv = bn_unpack(yq[u]);
                BF8 gv, ov;
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const bool on = NOY ? fmaf(xv.v[k], sc[k], sf[k]) > 0.f : yv.v[k] > 0.f;
                    gv.v[k] = on ? dv.v[k] : 0.f;
                    ov.v[k] = sc[k] * (gv.v[k] - k1[k] - (xv.v[k] - mu[k]) * rs[k] * k2[k]);
                }
                dx[rr * G + g] = bn_pack(ov);
                if (dskip) dskip[rr * G + g] = bn_pack(gv);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------
// launchers.  Workspace (floats): part[grid][2][C] | scale[C] | shift[C] (forward) or c1[C] | c2[C]
// ---------------------------------------------------------------------------------------
static int bn_grid() {
    static int grid = 0;
    if (!grid) {
        int dev = 0, sms = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        grid = (sms > 0 ? sms : 148) * 8;                  // 8 resident blocks of 256 threads per SM
    }
    return grid;
}

size_t bb_bn_workspace_floats(int C) { return (size_t)bn_grid() * 2 * C + 2 * (size_t)C; }

cudaError_t bb_launch_bn_relu_fwd(const void* x, const void* skip, const float* gamma, const float* beta,
                                  const float* pre_bias, float* running_mean, float* running_var, float momentum, float eps, int training,
                                  void* y, float* save_mean, float* save_rstd, float* workspace, int64_t M, int C,
                                  cudaStream_t stream) {
    const int grid = bn_grid();
    float* part = workspace;
    float* scale = workspace + (size_t)grid * 2 * C;
    float* shift = scale + C;
    const int R = BN_THREADS / (C >> 3);
    const int64_t need = (M + R - 1) / R;
    const int g = (int)(need < grid ? need : grid);
    if (training) {
        bb_bn_reduce_kernel<0><<<g, BN_THREADS, (size_t)R * 2 * C * sizeof(float), stream>>>(
            (const uint4*)x, nullptr, nullptr, nullptr, nullptr, part, M, C);
        bb_bn_finalize_fwd_kernel<<<C, BN_FIN_THREADS, 0, stream>>>(part, g, M, C, eps, momentum, gamma, beta, pre_bias,
                                                                      running_mean, running_var, save_mean, save_rstd, scale, shift,
                                                                      (const __nv_bfloat16*)x);
    } else {
        bb_bn_affine_eval_kernel<<<(C + 127) / 128, 128, 0, stream>>>(gamma, beta, pre_bias, running_mean, running_var, eps, C, scale, shift);
    }
    const int64_t need4 = (need + 3) / 4;
    bb_bn_apply_kernel<<<(int)(need4 < grid ? (need4 > 0 ? need4 : 1) : grid), BN_THREADS, 0, stream>>>(
        (const uint4*)x, (const uint4*)skip, scale, shift, (uint4*)y, M, C);
    return cudaGetLastError();
}

static inline int64_t noy_rows(int64_t need, bool noy) { return noy ? (need + 2) / 3 : (need + 1) / 2; }   // blocks for U rows per trip

cudaError_t bb_launch_bn_relu_bwd(const void* x, const void* y, const void* dy, const float* gamma,
                                  const float* save_mean, const float* save_rstd, void* dx, void* dskip,
                                  float* dgamma, float* dbeta, float* workspace, int64_t M, int C, cudaStream_t stream,
                                  const float* beta) {
    const int grid = bn_grid();
    float* part = workspace;
    float* c1 = workspace + (size_t)grid * 2 * C;
    float* c2 = c1 + C;
    const int R = BN_THREADS / (C >> 3);
    const int64_t need = (M + R - 1) / R;
    const int g = (int)(need < grid ? need : grid);
    const bool noy = y == nullptr;        // no residual input: the mask comes from x (needs beta)
    if (noy)
        bb_bn_reduce_kernel<2><<<g, BN_THREADS, (size_t)R * 2 * C * sizeof(float), stream>>>(
            (const uint4*)x, nullptr, (const uint4*)dy, save_mean, save_rstd, part, M, C, gamma, beta);
    else
        bb_bn_reduce_kernel<1><<<g, BN_THREADS, (size_t)R * 2 * C * sizeof(float), stream>>>(
            (const uint4*)x, (const uint4*)y, (const uint4*)dy, save_mean, save_rstd, part, M, C);
    bb_bn_finalize_bwd_kernel<<<C, BN_FIN_THREADS, 0, stream>>>(part, g, M, C, dgamma, dbeta, c1, c2);
    const int64_t need2 = noy_rows(need, y == nullptr);
    const int gdx = (int)(need2 < grid ? (need2 > 0 ? need2 : 1) : grid);
    if (noy)
        bb_bn_dx_kernel<true><<<gdx, BN_THREADS, 0, stream>>>(
            (const uint4*)x, nullptr, (const uint4*)dy, save_mean, save_rstd, gamma, c1, c2, (uint4*)dx, (uint4*)dskip, M, C, beta);
    else
        bb_bn_dx_kernel<false><<<gdx, BN_THREADS, 0, stream>>>(
            (const uint4*)x, (const uint4*)y, (const uint4*)dy, save_mean, save_rstd, gamma, c1, c2, (uint4*)dx, (uint4*)dskip, M, C);
    return cudaGetLastError();
}
