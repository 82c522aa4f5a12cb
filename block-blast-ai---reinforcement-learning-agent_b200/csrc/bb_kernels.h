// bb_kernels.h — internal declarations shared by the kernel translation units and the C ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "bb_rules.cuh"

#ifndef BB_STEP_THREADS
#define BB_STEP_THREADS 256
#endif
#ifndef BB_STEP_MIN_BLOCKS
#define BB_STEP_MIN_BLOCKS 3
#endif

// device-side view of a batch of envs (SoA of 16-byte words, see bb_rules.cuh BBState)
struct BBEnvArrays {
    uint4* s0;   // board lo, board hi, pieces, aux
    uint4* s1;   // score, streak, moves, lines_total
    uint4* s2;   // max_streak, blocks_total, draw_ctr, policy_ctr
    int64_t n;
    int64_t env_offset;   // global id of env 0 of this shard
    uint64_t seed;
    uint32_t flags;
    BBEpisodeEnd* ep_end;   // optional [n] records written where an env terminates (bb_env_set_episode_end_buffer)
    int64_t out_stride;     // plane stride of mask outputs; 0 = n (set when a launch covers a sub-range of the envs)
    const uint8_t* trios;   // injected candidate trios [n][trio_len][3] (bb_env_set_trios) or NULL = Philox
    int64_t trio_len;
    int64_t trio_base;      // global id of the env that owns row 0 of `trios`
};

cudaError_t bb_launch_step(const BBEnvArrays& E, const BBRewardCfg& cfg, const int32_t* actions,
                           float* rewards, uint8_t* terminated, uint64_t* mask_out, uint64_t* board_out,
                           uint32_t* pieces_out, int32_t* ep_score, int32_t* ep_len, uint32_t* info_out,
                           unsigned long long* stats, cudaStream_t stream);
// one step of envs [off, off + cnt) only (the host-buffer entry point pipelines chunks of the batch
// against their device-to-host copies); output pointers are those of the WHOLE batch
cudaError_t bb_launch_step_range(const BBEnvArrays& E, const BBRewardCfg& cfg, int64_t off, int64_t cnt,
                                 const int32_t* actions, float* rewards, uint8_t* terminated, uint64_t* mask_out,
                                 int32_t* ep_score, int32_t* ep_len, uint32_t* info_out, uint64_t* board_out,
                                 uint32_t* pieces_out, cudaStream_t stream);
cudaError_t bb_launch_step_random(const BBEnvArrays& E, const BBRewardCfg& cfg, int n_steps, int per_step,
                                  int32_t* actions_out, float* rewards, uint8_t* terminated,
                                  uint64_t* mask_out, unsigned long long* stats, const uint64_t* mask_in,
                                  cudaStream_t stream);
cudaError_t bb_launch_zero_draw_ctr(const BBEnvArrays& E, cudaStream_t stream);
cudaError_t bb_launch_reset(const BBEnvArrays& E, const uint8_t* reset_mask, uint64_t* mask_out, cudaStream_t stream);
cudaError_t bb_launch_sample_valid(const BBEnvArrays& E, uint64_t call_counter, int32_t* actions_out, cudaStream_t stream);
// bb_env_expand (phase 1 + phase 2); scratch: bb_expand_scratch_count(n) int64 block totals (+ one grand total)
int64_t bb_expand_scratch_count(int64_t n);
// bb_env_observe_live; scratch: the same bb_expand_scratch_count(n) int64
cudaError_t bb_launch_observe_live(const BBEnvArrays& E, int64_t* scratch, uint64_t* board_out, uint32_t* pieces_out,
                                   uint64_t* mask_out, int64_t mask_stride, int32_t* ids_out, int32_t* count_out,
                                   cudaStream_t stream);
cudaError_t bb_launch_expand(const BBEnvArrays& E, const BBRewardCfg& cfg, uint32_t call_counter, int samples,
                             int64_t capacity, int64_t* offsets, int64_t* scratch, int32_t* action_out, float* reward_out,
                             uint8_t* terminated_out, uint32_t* info_out, uint64_t* board_out, uint32_t* pieces_out,
                             uint64_t* mask_out, cudaStream_t stream);
cudaError_t bb_launch_observe(const BBEnvArrays& E, uint64_t* board_out, uint32_t* pieces_out,
                              uint64_t* mask_out, cudaStream_t stream);

cudaError_t bb_launch_unpack_obs(const uint64_t* board, const uint32_t* pieces, const uint64_t* mask,
                                 int64_t mask_stride, void* obs_nchw, int obs_dtype, void* mask_dense,
                                 int mask_dtype, int64_t n, cudaStream_t stream, void* pieces_split = nullptr);
cudaError_t bb_launch_gather_minibatch(const int64_t* index, int64_t B, int64_t N, const uint64_t* board,
                                       const uint32_t* pieces, const uint64_t* mask, const int32_t* action,
                                       const float* logp, const float* adv, const float* ret, const float* mean_std,
                                       void* obs, int obs_dtype, uint64_t* mask_out, int32_t* action_out, float* logp_out,
                                       float* adv_out, float* ret_out, cudaStream_t stream);
// K7a (eight views of each row, view-major; index: optional row gather) and K7b (view average of the logits)
cudaError_t bb_launch_unpack_obs_sym(const uint64_t* board, const uint32_t* pieces, const int64_t* index, void* obs,
                                     int obs_dtype, int64_t n, cudaStream_t stream);
cudaError_t bb_launch_sym_logits_mean(const void* logits, int dtype, const uint32_t* pieces, float* out, int64_t n,
                                      cudaStream_t stream);
cudaError_t bb_launch_sym_logits_mean_bwd(const float* dout, const uint32_t* pieces, void* dlogits, int dtype, int64_t n,
                                          cudaStream_t stream);
// K7c (canonical view of each row and its view set; index: optional row gather) and the map of the canonical
// row's logits into the state's own frame, with its transpose
cudaError_t bb_launch_sym_canonical(const uint64_t* board, const uint32_t* pieces, const int64_t* index, uint64_t* cboard,
                                    uint32_t* cpieces, uint8_t* views, int64_t n, cudaStream_t stream);
cudaError_t bb_launch_sym_logits_canonical(const void* logits, int dtype, const uint32_t* pieces, const uint8_t* views,
                                           float* out, int64_t n, cudaStream_t stream);
cudaError_t bb_launch_sym_logits_canonical_bwd(const float* dout, const uint32_t* pieces, const uint8_t* views, void* dlogits,
                                               int dtype, int64_t n, cudaStream_t stream);
cudaError_t bb_launch_masked_sample(const void* logits, int logits_dtype, const uint64_t* mask,
                                    int64_t mask_stride, uint64_t seed, uint64_t call_counter, int mode,
                                    int32_t* action, float* logp, float* entropy, int64_t n, cudaStream_t stream,
                                    int64_t row_offset = 0, const uint64_t* counter_dev = nullptr);
cudaError_t bb_launch_masked_head_bwd(const void* logits, int dtype, const uint64_t* mask, int64_t mask_stride,
                                      const int32_t* action, const float* g_logp, const float* g_ent,
                                      void* dlogits, int64_t n, cudaStream_t stream);
cudaError_t bb_launch_ppo_loss(const void* logits, int dtype, const uint64_t* mask, int64_t mask_stride,
                               const int32_t* action, const float* old_logp, const float* adv, const float* ret,
                               const float* value, float clip, float value_coef, float entropy_coef,
                               void* dlogits, float* dvalue, double* sums, int64_t n, cudaStream_t stream);
cudaError_t bb_launch_gae(const float* rewards, const float* values, const float* dones,
                          const float* last_values, float gamma, float gamma_lam, float* adv, float* ret,
                          double* moments, int64_t T, int64_t N, cudaStream_t stream);
size_t bb_bn_workspace_floats(int C);
cudaError_t bb_launch_bn_relu_fwd(const void* x, const void* skip, const float* gamma, const float* beta,
                                  const float* pre_bias, float* running_mean, float* running_var, float momentum, float eps, int training,
                                  void* y, float* save_mean, float* save_rstd, float* workspace, int64_t M, int C,
                                  cudaStream_t stream);
cudaError_t bb_launch_bn_relu_bwd(const void* x, const void* y, const void* dy, const float* gamma,
                                  const float* save_mean, const float* save_rstd, void* dx, void* dskip,
                                  float* dgamma, float* dbeta, float* workspace, int64_t M, int C, cudaStream_t stream,
                                  const float* beta = nullptr);   // y == NULL: ReLU mask recomputed from x (needs beta)
