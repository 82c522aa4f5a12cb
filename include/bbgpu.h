/* bbgpu.h — C ABI of libbbgpu.so: B200 (sm_100a) batched Block Blast simulator and the
 * masked-PPO rollout kernels.
 *
 * The reference (rfahd1525/Block-Blast-AI---Reinforcement-Learning-Agent) is pure Python and
 * has no FFI; its boundary for this path is the Python class API.  Each entry point below
 * names the reference interface it replaces (file:line in the reference checkout); the
 * Python mirror of those classes lives in block-blast-ai---reinforcement-learning-agent_b200/
 * and INTEGRATION.md shows the ctypes stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error; bb_last_error() gives the message of
 *     the last failure on the calling thread.  No exceptions, no aborts.
 *   - pointers documented "device" are CUDA device pointers owned by the caller (e.g. torch
 *     tensors); the library never frees or retains them after the call returns.
 *   - `stream` is a cudaStream_t passed as void* (torch.cuda.current_stream().cuda_stream);
 *     calls are asynchronous on it, never synchronise, and never allocate after create
 *     (except the *_host entry points, which copy and synchronise).
 *   - a bb_env lives on the CUDA device current at bb_env_create time; calls made with another
 *     device current are refused (error code -1); it is not thread-safe.
 *   - bit convention for boards and masks: bit = row*8 + col; action = piece*64 + row*8 + col
 *     (src/environment/block_blast_env.py:104-132).
 *   - action masks are three bit-planes per env stored plane-major: mask[p*n_envs + i].
 *   - packed pieces word: bytes 0..2 = piece indices (PIECE_LIST order,
 *     src/game/pieces.py:244-318), byte 3 = used bits (bit p set = piece p already placed).
 *   - invalid actions are NOT errors: reward -10, state untouched (block_blast_env.py:240-245).
 */
#ifndef BBGPU_H
#define BBGPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BB_ABI_VERSION 2

/* flags for bb_env_create */
#define BB_ENV_RESEED_ON_RESET 1u /* every reset restarts the env's trio stream: the reference's
                                     behaviour when a seed is given (wrappers.py:102 ->
                                     block_blast_env.py:215 -> engine.py:137-138) */
#define BB_ENV_NO_AUTO_RESET 2u   /* single-env semantics (BlockBlastEnv.step): stay GAME_OVER */

/* dtype codes for dense outputs */
#define BB_F32 0
#define BB_BF16 1
#define BB_U8 2

typedef struct bb_env bb_env;

int bb_version(void);
const char* bb_last_error(void);

/* The 37-piece tables compiled into the kernels, for cross-checking against
 * src/game/pieces.py:78-318.  Host pointers; any may be NULL. */
int bb_piece_table(uint64_t* masks37, uint64_t* inb37, uint8_t* nblk37);

/* VectorizedBlockBlastEnv.__init__ (src/environment/wrappers.py:21-50) + the first reset.
 * reward_cfg = {line_clear_base, block_placed, game_over_penalty, hole_penalty, center_bonus,
 * combo_multiplier_bonus, survival_bonus} (block_blast_env.py:63-71); NULL = defaults.
 * Env i draws candidate trios from Philox stream (seed, global_env_offset + i), so a shard on
 * any GPU reproduces the same trajectories as the single-GPU run. */
int bb_env_create(bb_env** out, int64_t n_envs, uint64_t seed, int64_t global_env_offset,
                  const double reward_cfg[7], uint32_t flags);
int bb_env_destroy(bb_env* env);
int64_t bb_env_num_envs(const bb_env* env);

/* Optional episode-end log: `records` is a device array of n_envs 32-byte records
 *   {u64 board; u32 pieces; i32 lines_total, max_streak, blocks_total; u32 holes | filled<<8;
 *    u32 last_move (the info word of the terminal move)}
 * Record i is written by every later step call in which env i terminates, with the TERMINAL
 * state (before the auto-reset): what the reference leaves in infos[i] for a finished episode
 * (block_blast_env.py:266-288, wrappers.py:97-100).  The pointer is retained until replaced;
 * NULL switches the log off.  This is the only pointer the library keeps between calls. */
int bb_env_set_episode_end_buffer(bb_env* env, void* records);

/* Injected candidate trios — the replay / parity mode ("fed the same piece sequences").
 * h_trios: HOST u8[n_envs][len][3], piece indices in [0,37): entry [i][d] is what the reference's
 * engine.rng.choice(37, size=3, replace=True) (src/game/pieces.py:350-355, called from
 * GameEngine._generate_new_pieces, src/game/engine.py:155-172) returns for env i at its d-th call.
 * The table replaces the env's Philox stream: candidate number d of env i is h_trios[i][d % len],
 * accepted or rejected by the same solvability rule.  The library keeps its own device copy, sets
 * every env's draw counter to 0 and synchronises; call bb_env_reset afterwards to start episodes
 * on the new stream.  With BB_ENV_RESEED_ON_RESET every reset restarts at entry 0, which is the
 * reference's behaviour for a seeded env (numpy's PCG64 re-seeded on every reset, engine.py:137-138).
 * h_trios == NULL returns to the Philox streams. */
int bb_env_set_trios(bb_env* env, const uint8_t* h_trios, int64_t len, void* stream);

/* VectorizedBlockBlastEnv.reset (wrappers.py:53-73).  reset_mask: device u8[n] or NULL (= all).
 * mask_out: device u64[3*n] or NULL. */
int bb_env_reset(bb_env* env, const uint8_t* reset_mask, uint64_t* mask_out, void* stream);

/* VectorizedBlockBlastEnv.step (wrappers.py:75-116): BlockBlastEnv.step
 * (block_blast_env.py:224-264) -> GameEngine.make_move (src/game/engine.py:390-454) with
 * auto-reset.  One fused kernel: validate, place, clear rows/cols, score+streak, trio
 * regeneration (Philox + the "all three placeable" search, engine.py:155-238), game over,
 * shaped reward (block_blast_env.py:148-193), auto-reset, next action mask.
 *   actions     device i32[n]
 *   rewards     device f32[n]
 *   terminated  device u8[n]
 *   mask_out    device u64[3*n]   action mask of the state after the step     (may be NULL)
 *   board_out   device u64[n]     packed next observation: board               (may be NULL)
 *   pieces_out  device u32[n]     packed next observation: pieces word         (may be NULL)
 *   ep_score    device i32[n]     written only where terminated: info['final_score'] (NULL ok)
 *   ep_len      device i32[n]     written only where terminated: info['moves']       (NULL ok)
 *   info_out    device u32[n]     bit0 invalid_action, bits1-3 lines_cleared, bits4-7
 *                                 blocks_placed, bits8-10 combo_multiplier, bits11-17 candidate
 *                                 trios drawn, bits18-31 score_gained           (NULL ok)
 *   stats       device u64[5]     accumulated with atomics (NULL ok): env-steps, finished episodes,
 *                                 sum of their final scores, sum of their lengths, max final score —
 *                                 the episode statistics scripts/train.py:196-201 collects from infos
 */
int bb_env_step(bb_env* env, const int32_t* actions, float* rewards, uint8_t* terminated,
                uint64_t* mask_out, uint64_t* board_out, uint32_t* pieces_out, int32_t* ep_score,
                int32_t* ep_len, uint32_t* info_out, uint64_t* stats, void* stream);

/* n_steps of the same step with the uniform-random-valid-action policy of
 * sample_valid_actions (wrappers.py:133-136, block_blast_env.py:318-323) fused in: the action
 * is the k-th set bit of the 192-bit mask, k = mulhi(philox_word, n_valid).  State stays in
 * registers across the n_steps.  Outputs (all may be NULL) describe the LAST step;
 * stats: device u64[5] accumulated with atomics: env-steps, episodes, sum of final scores,
 * sum of episode lengths, max final score.
 * mask_in (device u64[3*n] or NULL): the action mask of the CURRENT states exactly as the previous
 * step / reset call wrote it to its mask_out (it may be the same buffer as mask_out) — the policy
 * then reads the observation it was given instead of recomputing it from the boards. */
int bb_env_step_random(bb_env* env, int32_t n_steps, int32_t* actions_out, float* rewards,
                       uint8_t* terminated, uint64_t* mask_out, uint64_t* stats,
                       const uint64_t* mask_in, void* stream);

/* Random-policy ROLLOUT: the same n_steps as bb_env_step_random in one launch (state in
 * registers), but every step's outputs are written: actions_out i32[n_steps][n], rewards
 * f32[n_steps][n], terminated u8[n_steps][n], mask_out u64[n_steps][3][n] (mask of the state
 * AFTER that step); any may be NULL.  Row t equals what bb_env_step_random(1) would have
 * produced at step t.  The data-collection form of the sample_valid_actions + step loop
 * (scripts/benchmark.py:127-129). */
int bb_env_rollout_random(bb_env* env, int32_t n_steps, int32_t* actions_out, float* rewards,
                          uint8_t* terminated, uint64_t* mask_out, uint64_t* stats, void* stream);

/* VectorizedBlockBlastEnv.sample_valid_actions (wrappers.py:133-136, block_blast_env.py:318-323):
 * one uniformly random valid action per env (0 if none), k-th set bit of the mask with
 * k = mulhi(philox_word, n_valid) on Philox stream 3 keyed by (seed, global env id, call_counter).
 * The env state is not modified.  actions_out: device i32[n] or NULL; h_actions_out: HOST
 * i32[n] or NULL (copies and synchronises when given).  At least one must be non-NULL. */
int bb_env_sample_valid_actions(bb_env* env, uint64_t call_counter, int32_t* actions_out,
                                int32_t* h_actions_out, void* stream);

/* One-ply look-ahead: every legal successor of every env's CURRENT state, without changing any
 * state (no counter moves either).  What a planner would otherwise get from GameEngine.make_move
 * (engine.py:390-454) on a copy of the engine per legal action, with _generate_new_pieces
 * (engine.py:155-172) and BlockBlastEnv._calculate_reward (block_blast_env.py:148-193).
 * Items of env i, in order: its valid actions in np.where(mask) order (piece 0's bits, then 1's,
 * then 2's: the order bb_env_sample_valid_actions indexes).  An action that does not use the last
 * unused piece gives ONE item: exactly what bb_env_step with that action returns for env i created
 * with BB_ENV_NO_AUTO_RESET.  When exactly one piece is left, every valid action deals a new trio and
 * gives `samples` items k = 0..samples-1 (k ascending): the same step, but the trio is dealt from the
 * LOOKAHEAD stream, NOT the env's own candidate stream (which would reveal the trio the env will
 * really be dealt): Philox key seed, counter (global env id lo, hi, call_counter << 7 | d,
 * 4 | k << 8), d = candidate 0..99 of the deal, piece ids mulhi(word, 37) of words 0..2, first solvable
 * candidate kept (the 100th when none is).  It does not depend on the action, so all deal items of
 * an env with the same k see the same candidates.  Game-over envs have no items.
 *   call_counter  < 2^25; samples 1..64; capacity >= 0 = room of the item arrays
 *   offsets        device i64[n+1]   exclusive scan of the item counts; offsets[n] = total.
 *                                    ALWAYS written completely (capacity 0 = size query)
 *   action_out     device i32[cap]   (every item array may be NULL; items >= capacity are dropped)
 *   reward_out     device f32[cap]   bit-exact bb_env_step reward
 *   terminated_out device u8[cap]
 *   info_out       device u32[cap]   bb_env_step's info word; candidates drawn = LOOKAHEAD draws
 *   board_out      device u64[cap]   successor board
 *   pieces_out     device u32[cap]   successor pieces word
 *   mask_out       device u64[3*cap] successor action mask, plane-major with plane stride `capacity`
 *                                    (all zero when terminated)
 * The same call_counter gives the same items, so a size query followed by a fill call is consistent. */
int bb_env_expand(bb_env* env, uint64_t call_counter, int32_t samples, int64_t capacity,
                  int64_t* offsets, int32_t* action_out, float* reward_out, uint8_t* terminated_out,
                  uint32_t* info_out, uint64_t* board_out, uint32_t* pieces_out, uint64_t* mask_out,
                  void* stream);

/* Packed observation of the current states (engine.get_observation, engine.py:478-507):
 * board_out device u64[n], pieces_out device u32[n], mask_out device u64[3*n]; any NULL. */
int bb_env_observe(bb_env* env, uint64_t* board_out, uint32_t* pieces_out, uint64_t* mask_out,
                   void* stream);

/* Packed observation of the envs that are NOT game over, compacted: row r = the r-th such env in
 * ascending env order, with exactly the bytes bb_env_observe writes for that env.  count_out[0] =
 * number of rows, written on the device (no host synchronisation); the rows are ordered without
 * atomics (per-block counts, a scan, the write), so a repeated call writes the same bytes.  Uses the
 * handle's create-time scratch, so two calls on one handle must not run concurrently.  No env state
 * changes.  Rows >= count_out[0] are left untouched.
 *   board_out  device u64[n]   pieces_out device u32[n]   ids_out device i32[n] (env index 0..n-1)
 *   mask_out   device u64[3*mask_stride], plane-major with plane stride mask_stride >= n
 *   count_out  device i32[1]
 * Every output is required. */
int bb_env_observe_live(bb_env* env, uint64_t* board_out, uint32_t* pieces_out, uint64_t* mask_out,
                        int64_t mask_stride, int32_t* ids_out, int32_t* count_out, void* stream);

/* Full state export / import for checkpoints and parity tests (GameEngine.get_state /
 * set_state, engine.py:456-476, plus counters).  HOST arrays of n_envs records, 48 bytes each:
 * {u64 board; u32 pieces; u32 aux(prev_holes | prev_center_filled<<8 | game_over<<16);
 *  i32 score, streak, moves, lines_total, max_streak, blocks_total; u32 draw_ctr, policy_ctr}.
 * Synchronises the stream. */
int bb_env_get_state(bb_env* env, void* host_records, void* stream);
int bb_env_set_state(bb_env* env, const void* host_records, void* stream);

/* Same as bb_env_step but with HOST buffers (pinned memory recommended): copies actions to
 * the device, steps, copies rewards/terminated/packed obs back, synchronises.  This is the
 * call the numpy-facing VectorizedBlockBlastEnv.step makes.  board/pieces/mask/ep_* may be
 * NULL to skip that copy; h_info receives the per-env info word of bb_env_step.
 * bb_env_host_layout gives byte offsets {mask, board, rewards, pieces, ep_score, ep_len, info,
 * terminated} into ONE host block: mask/board/rewards/pieces/terminated form a prefix of
 * prefix_bytes (41 B/env rounded up to 16), ep_score/ep_len/info follow.  When the host arrays sit
 * at these offsets the results come back in a single transfer: 41 B/env when the three tail
 * arrays are NULL, 53 B/env when they are given.  The tail of the LAST host step stays on the
 * device and can be fetched on demand with bb_env_fetch_step_info (the training loop reads
 * infos of terminated envs only, scripts/train.py:196-201). */
int bb_env_host_layout(int64_t n_envs, int64_t offsets8[8], int64_t* total_bytes, int64_t* prefix_bytes);
int bb_env_step_host(bb_env* env, const int32_t* h_actions, float* h_rewards,
                     uint8_t* h_terminated, uint64_t* h_board, uint32_t* h_pieces,
                     uint64_t* h_mask, int32_t* h_ep_score, int32_t* h_ep_len, uint32_t* h_info,
                     void* stream);
int bb_env_fetch_step_info(bb_env* env, int32_t* h_ep_score, int32_t* h_ep_len, uint32_t* h_info,
                           void* stream);

/* The host-buffer step in the REFERENCE'S OWN observation layout, for callers that read the dense
 * arrays every step (wrappers.py:110-126 returns them; PPOAgent.select_actions reads them):
 * h_block is one HOST block laid out by bb_env_host_dense_layout, byte offsets {board f32[n][8][8],
 * pieces f32[n][3][8][8], action_mask i8[n][192], rewards f32[n], terminated u8[n]} = 1,221 B/env.
 * The observation is expanded on the device (K2) and arrives in ONE transfer; the packed
 * observation and the info arrays of the step stay in the device staging block
 * (bb_env_fetch_step_info).  bb_env_observe_host_dense fills the same block for the current
 * states without stepping (reset; rewards / terminated are left untouched). */
int bb_env_host_dense_layout(int64_t n_envs, int64_t offsets5[5], int64_t* total_bytes);
int bb_env_step_host_dense(bb_env* env, const int32_t* h_actions, void* h_block, void* stream);
int bb_env_observe_host_dense(bb_env* env, void* h_block, void* stream);

/* Observation expansion (engine.get_observation + Piece.to_mask, engine.py:489-507,
 * src/game/pieces.py:39-45; network input cat([board, pieces]), src/models/network.py:152-158).
 *   board device u64[n], pieces device u32[n], mask device u64[3*n] plane-major with plane
 *   stride mask_stride (elements)
 *   obs_nchw    device [n,4,8,8] of obs_dtype (BB_F32 / BB_BF16); NULL to skip
 *   mask_dense  device [n,192] of mask_dtype (BB_U8 / BB_F32);  NULL to skip */
int bb_unpack_obs(const uint64_t* board, const uint32_t* pieces, const uint64_t* mask,
                  int64_t mask_stride, void* obs_nchw, int obs_dtype, void* mask_dense,
                  int mask_dtype, int64_t n, void* stream);

/* The same expansion into the reference's three separate arrays (wrappers.py:118-126):
 * board_f32 device f32[n][8][8], pieces_f32 device f32[n][3][8][8], action_mask_i8 device
 * i8[n][192] (NULL to skip). */
int bb_unpack_obs_reference_layout(const uint64_t* board, const uint32_t* pieces, const uint64_t* mask,
                                   int64_t mask_stride, float* board_f32, float* pieces_f32,
                                   int8_t* action_mask_i8, int64_t n, void* stream);

/* Minibatch assembly of the PPO update (RolloutBuffer.get_samples, src/agents/ppo.py:171-213: the
 * reference flattens the (T, N) buffer, normalises the advantages and gathers seven arrays by a
 * random permutation).  Row b of the minibatch is sample index[b] (flat t*n_envs + e) of the
 * packed device-resident rollout buffer:
 *   index device i64[batch]; board device u64[T*n_envs]; pieces device u32[T*n_envs];
 *   mask device u64[T][3][n_envs]; action i32, logp / adv / ret f32 [T*n_envs]
 *   adv_mean_std device f32[2] or NULL: adv_out = (adv - mean) / (std + 1e-8) (ppo.py:196)
 *   obs_nchw device [batch,4,8,8] of obs_dtype, or NULL to gather everything but the observation
 *            planes (obs_dtype is then ignored); mask_out device u64[3][batch];
 *   action_out i32, logp_out / adv_out / ret_out f32 [batch] */
int bb_gather_minibatch(const int64_t* index, int64_t batch, int64_t n_envs, const uint64_t* board,
                        const uint32_t* pieces, const uint64_t* mask, const int32_t* action,
                        const float* logp, const float* adv, const float* ret,
                        const float* adv_mean_std, void* obs_nchw, int obs_dtype, uint64_t* mask_out,
                        int32_t* action_out, float* logp_out, float* adv_out, float* ret_out,
                        void* stream);

/* Board symmetries (group D4, ids and maps in csrc/bb_rules.cuh): the symmetric policy evaluates
 * the network on the eight views of each state and averages over them.
 * bb_unpack_obs_sym: the observation planes of bb_unpack_obs for all eight views, view-major:
 *   row g*n + i of obs_nchw device [8n,4,8,8] of obs_dtype (BB_F32 / BB_BF16) is view g of input
 *   row index[i] (index device i64[n], or NULL for row i) of board device u64[], pieces device u32[].
 * bb_sym_logits_mean: out device f32[n,192],
 *   out[i, s*64 + a] = 0.125 * sum_{g=0..7} logits[g*n + i, s*64 + sigma_{g,p_s}(a)]
 *   (f32 sum in g order) where a is an in-bounds anchor of the piece p_s < 37 of slot s of
 *   pieces[i] (device u32[n]), 0 elsewhere.  logits device [8n,192] of logits_dtype, raw, 16-byte
 *   aligned (read as 16-byte vectors; an unaligned pointer is rejected with code -1).
 * bb_sym_logits_mean_backward: the transposed map, grad_logits device [8n,192] of logits_dtype:
 *   0.125 * grad_out[i, s*64 + a] at the view position of every such (s, a), 0 elsewhere;
 *   grad_logits 16-byte aligned like logits. */
int bb_unpack_obs_sym(const uint64_t* board, const uint32_t* pieces, const int64_t* index, void* obs_nchw,
                      int obs_dtype, int64_t n, void* stream);
int bb_sym_logits_mean(const void* logits, int logits_dtype, const uint32_t* pieces, float* out, int64_t n,
                       void* stream);
int bb_sym_logits_mean_backward(const float* grad_out, const uint32_t* pieces, void* grad_logits,
                                int logits_dtype, int64_t n, void* stream);

/* Canonical frame (group D4 as above): the network runs once per state, on the canonical view of its orbit,
 * and its logits are mapped back into the state's own frame; policy and value are then exactly invariant /
 * equivariant under the eight symmetries at the cost of one network row per state.
 * bb_sym_canonical: for row r = index[i] (index device i64[n], or NULL for r = i) of board device u64[],
 *   pieces device u32[]: board_out / pieces_out device u64[n] / u32[n] = the view g (bb_sym_board(g, b),
 *   bb_sym_pieces(g, pw)) with the smallest key (board as u64, then the full pieces word as u32), and
 *   views_out device u8[n] = the view set M: bit g set iff view g equals that view (never 0).
 * bb_sym_logits_canonical: out device f32[n,192],
 *   out[i, s*64 + a] = (1/|M_i|) * sum_{g in M_i, ascending} logits[i, s*64 + sigma_{g,p_s}(a)]
 *   (f32) where a is an in-bounds anchor of the piece p_s < 37 of slot s of the state's own pieces[i]
 *   (device u32[n]), 0 elsewhere.  logits device [n,192] of logits_dtype: the network's raw logits of
 *   the canonical rows, 16-byte aligned (an unaligned pointer is rejected with code -1); views device
 *   u8[n] from bb_sym_canonical.
 * bb_sym_logits_canonical_backward: the transposed map, grad_logits device [n,192] of logits_dtype:
 *   each canonical position sums (1/|M|) * grad_out over the (g, s*64 + a) that reach it, in ascending g
 *   (several when |M| > 1), 0 where none does; grad_out device f32[n,192]; both 16-byte aligned. */
int bb_sym_canonical(const uint64_t* board, const uint32_t* pieces, const int64_t* index, uint64_t* board_out,
                     uint32_t* pieces_out, uint8_t* views_out, int64_t n, void* stream);
int bb_sym_logits_canonical(const void* logits, int logits_dtype, const uint32_t* pieces, const uint8_t* views,
                            float* out, int64_t n, void* stream);
int bb_sym_logits_canonical_backward(const float* grad_out, const uint32_t* pieces, const uint8_t* views,
                                     void* grad_logits, int logits_dtype, int64_t n, void* stream);

/* Masked categorical head (BlockBlastNetwork.forward masking + get_action_and_value +
 * _masked_entropy, src/models/network.py:172-262) fused in one kernel.
 *   logits  device [n,192] of logits_dtype (BB_F32 / BB_BF16), raw (unmasked)
 *   mask    device u64[3*n] plane-major, plane stride mask_stride
 *   mode 0: sample  action ~ softmax(masked logits) by inverse CDF on a Philox uniform
 *                   (SAMPLE stream: key seed, counter (row_offset + row, call_counter +
 *                   *call_counter_dev)); row_offset = global id of row 0, so env shards on
 *                   several GPUs draw independent noise; call_counter_dev (device u64, NULL = 0)
 *                   lets a captured CUDA graph advance the counter between replays
 *   mode 1: argmax  (deterministic=True)
 *   mode 2: evaluate the actions given in `action` (PPO update path)
 *   action   device i32[n]  (out for modes 0/1, in for mode 2)
 *   logp     device f32[n]  log(clamp(p/sum(p), eps, 1-eps))[action]  (torch Categorical)
 *   entropy  device f32[n]  masked entropy (network.py:232-262); NULL to skip */
int bb_masked_sample(const void* logits, int logits_dtype, const uint64_t* mask,
                     int64_t mask_stride, uint64_t seed, uint64_t call_counter, int mode,
                     int32_t* action, float* logp, float* entropy, int64_t n, int64_t row_offset,
                     const uint64_t* call_counter_dev, void* stream);

/* Backward of bb_masked_sample(mode 2) for the PPO update: autograd of log_prob[action] and the
 * masked entropy through softmax / Categorical (network.py:210-262 as differentiated at
 * src/agents/ppo.py:366-395).  grad_logits[n,192] (same dtype as logits) =
 *   grad_logp * [eps <= p_a <= 1-eps] * (onehot(action) - p)  -  grad_entropy * p * (log p + H),
 * zero at masked actions.  grad_entropy may be NULL. */
int bb_masked_head_backward(const void* logits, int logits_dtype, const uint64_t* mask,
                            int64_t mask_stride, const int32_t* action, const float* grad_logp,
                            const float* grad_entropy, void* grad_logits, int64_t n, void* stream);

/* The whole PPO loss tail of one minibatch in one pass over the logits (PPOAgent.update,
 * src/agents/ppo.py:366-395, with network.py:210-262 inside): masked log-softmax, log-prob of the
 * stored action, ratio to old_logp, clipped surrogate, value MSE and masked-entropy bonus;
 *   loss = mean(-min(r A, clip(r, 1-eps, 1+eps) A)) + value_coef mean((v-R)^2) - entropy_coef mean(H).
 * Writes grad_logits[n,192] (dtype of logits) and grad_values f32[n] = d loss / d(.), and ADDS to
 * sums5 (device f64[5], zero it first): sum of -min(..), (v-R)^2, H, (r-1)-log r, [|r-1| > eps];
 * divide by n for policy_loss, value_loss, entropy, approx_kl, clip_fraction. */
int bb_ppo_loss(const void* logits, int logits_dtype, const uint64_t* mask, int64_t mask_stride,
                const int32_t* action, const float* old_logp, const float* advantages,
                const float* returns, const float* values, double clip_epsilon, double value_coef,
                double entropy_coef, void* grad_logits, float* grad_values, double* sums5, int64_t n,
                void* stream);

/* BatchNorm2d + ReLU (+ residual add) of the policy CNN on channels-last bf16 activations
 * (src/models/network.py:14-31 ResidualBlock, :78-92 conv encoder: conv -> BatchNorm2d -> ReLU, and
 * conv -> BatchNorm2d -> "+ x" -> ReLU).  The convolutions stay cuDNN; these two calls replace
 * torch's batch_norm / relu / add kernels around them with HBM-roofline passes.
 *   x, skip, y, grad_*: device bf16 [rows, channels], rows = N*H*W (NHWC memory), channels % 8 == 0
 *   gamma, beta, running_*, save_*, grad_gamma, grad_beta: device f32 [channels]
 *   workspace: device f32 [bb_bn_workspace_size(channels)]
 * forward : training != 0: batch statistics (biased variance for the normalisation, running
 *           statistics updated with momentum and the unbiased variance like torch.nn.BatchNorm2d),
 *           save_mean / save_rstd written for backward; training == 0: running statistics.
 *           y = relu((x - mean) * rstd * gamma + beta (+ skip)); skip may be NULL.
 *           pre_bias (f32 [channels] or NULL): a per-channel constant the caller did NOT add to x
 *           — the bias of the convolution in front, which BatchNorm cancels in y — so the conv's
 *           bias-add and bias-gradient passes disappear; it is added to the tracked running mean
 *           (training) and to x (eval) so the module behaves exactly as conv(bias) -> BatchNorm.
 * backward: g = grad_y * [y > 0]; grad_beta = sum g; grad_gamma = sum g * xhat;
 *           grad_x = gamma * rstd * (g - mean(g) - xhat * mean(g * xhat)); grad_skip = g (NULL to skip). */
int64_t bb_bn_workspace_size(int channels);
int bb_bn_relu_forward(const void* x, const void* skip, const float* gamma, const float* beta,
                       const float* pre_bias, float* running_mean, float* running_var, double momentum, double eps,
                       int training, void* y, float* save_mean, float* save_rstd, float* workspace,
                       int64_t rows, int channels, void* stream);
int bb_bn_relu_backward(const void* x, const void* y, const void* grad_y, const float* gamma,
                        const float* save_mean, const float* save_rstd, void* grad_x, void* grad_skip,
                        float* grad_gamma, float* grad_beta, float* workspace, int64_t rows,
                        int channels, void* stream);

/* The backward pass of a layer WITHOUT a residual input (conv -> BatchNorm2d -> ReLU, network.py:78-92 and the first
 * half of ResidualBlock, :24-27): the ReLU mask [y > 0] is recomputed from x with the forward's own affine pair
 * (y = relu(x * gamma * rstd + (beta - mean * gamma * rstd))), so y is not read back: 5 activation passes instead of 7. */
int bb_bn_relu_backward_no_skip(const void* x, const void* grad_y, const float* gamma, const float* beta,
                                const float* save_mean, const float* save_rstd, void* grad_x, float* grad_gamma,
                                float* grad_beta, float* workspace, int64_t rows, int channels, void* stream);

/* GAE and returns (RolloutBuffer.compute_returns_and_advantages, src/agents/ppo.py:141-169),
 * reverse scan over T, float32, same operation order as the reference (bit-identical).
 *   rewards, values, dones: device f32[T*N] time-major; last_values device f32[N]
 *   adv, ret: device f32[T*N]
 *   moments: device f64[2] or NULL: += sum(adv), sum(adv^2)  (whole-buffer normalisation,
 *   ppo.py:196; all-reduce them across ranks) */
int bb_gae(const float* rewards, const float* values, const float* dones,
           const float* last_values, double gamma, double lam, float* adv, float* ret,
           double* moments, int64_t T, int64_t N, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BBGPU_H */
