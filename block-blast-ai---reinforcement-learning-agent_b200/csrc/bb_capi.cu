// bb_capi.cu — the extern "C" boundary declared in include/bbgpu.h.
// Plain pointers and sizes only; errors become return codes + a thread-local message.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <new>
#include "../../include/bbgpu.h"
#include "bb_kernels.h"

static thread_local char g_err[512] = "";

static int fail(int code, const char* what, cudaError_t e = cudaSuccess) {
    if (e != cudaSuccess) snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
    else snprintf(g_err, sizeof(g_err), "%s", what);
    return code;
}
#define BB_CUDA(call, what) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return fail(-2, what, e__); } while (0)
// every entry point that launches on an env's arrays runs with the env's device current
#define BB_DEVICE(e, what) do { int d__ = -1; cudaError_t e__ = cudaGetDevice(&d__); \
    if (e__ != cudaSuccess) return fail(-2, what, e__); \
    if (d__ != (e)->device) return fail(-1, what ": the env lives on another CUDA device than the current one"); } while (0)

struct bb_env {
    BBEnvArrays arr;
    BBRewardCfg cfg;
    int device;
    // lazily allocated device staging for the host-buffer entry point
    int32_t* d_actions;
    float* d_rewards;
    uint8_t* d_terminated;
    uint64_t* d_board;
    uint32_t* d_pieces;
    uint64_t* d_mask;
    int32_t* d_ep_score;
    int32_t* d_ep_len;
    uint32_t* d_info;
    uint8_t* d_block;      // the eight result arrays above live in this one allocation (bb_env_host_layout)
    uint8_t* d_dense;      // lazily allocated reference-layout result block (bb_env_host_dense_layout)
    uint8_t* d_trios;      // injected candidate trios (bb_env_set_trios), owned
    int64_t* d_expand_scratch;   // block totals of bb_env_expand's offset scan, sized by n_envs at create
};

static const double BB_DEFAULT_CFG[7] = {1.0, 0.01, -1.0, -0.05, 0.02, 0.5, 0.001};

extern "C" {

static int ensure_staging(bb_env* e);
static int ensure_dense(bb_env* e);

int bb_version(void) { return BB_ABI_VERSION; }
const char* bb_last_error(void) { return g_err; }

int bb_piece_table(uint64_t* masks37, uint64_t* inb37, uint8_t* nblk37) {
    for (int i = 0; i < BB_NUM_PIECES; ++i) {
        if (masks37) masks37[i] = BB_HOST_PIECE_MASKS[i];
        if (inb37) inb37[i] = BB_HOST_PIECE_INB[i];
        if (nblk37) nblk37[i] = (uint8_t)BB_META_N(BB_HOST_PIECE_META[i]);
    }
    return 0;
}

int bb_env_create(bb_env** out, int64_t n_envs, uint64_t seed, int64_t global_env_offset,
                  const double reward_cfg[7], uint32_t flags) {
    if (!out) return fail(-1, "bb_env_create: out is NULL");
    *out = nullptr;
    if (n_envs <= 0) return fail(-1, "bb_env_create: n_envs must be > 0");
    if (global_env_offset < 0) return fail(-1, "bb_env_create: negative global_env_offset");
    bb_env* e = new (std::nothrow) bb_env();
    if (!e) return fail(-3, "bb_env_create: out of host memory");
    memset(e, 0, sizeof(*e));
    cudaError_t err = cudaGetDevice(&e->device);
    if (err != cudaSuccess) {
        bb_env_destroy(e);
        return fail(-2, "bb_env_create: cudaGetDevice", err);
    }
    e->arr.n = n_envs;
    e->arr.env_offset = global_env_offset;
    e->arr.trio_base = global_env_offset;
    e->arr.seed = seed;
    e->arr.flags = flags;
    const double* c = reward_cfg ? reward_cfg : BB_DEFAULT_CFG;
    e->cfg.line_clear_base = c[0]; e->cfg.block_placed = c[1]; e->cfg.game_over_penalty = c[2];
    e->cfg.hole_penalty = c[3]; e->cfg.center_bonus = c[4]; e->cfg.combo_multiplier_bonus = c[5];
    e->cfg.survival_bonus = c[6];
    const size_t bytes = (size_t)n_envs * sizeof(uint4);
    if ((err = cudaMalloc(&e->arr.s0, bytes)) != cudaSuccess || (err = cudaMalloc(&e->arr.s1, bytes)) != cudaSuccess ||
        (err = cudaMalloc(&e->arr.s2, bytes)) != cudaSuccess) {
        bb_env_destroy(e);
        return fail(-2, "bb_env_create: cudaMalloc state", err);
    }
    if ((err = cudaMemset(e->arr.s0, 0, bytes)) != cudaSuccess || (err = cudaMemset(e->arr.s1, 0, bytes)) != cudaSuccess ||
        (err = cudaMemset(e->arr.s2, 0, bytes)) != cudaSuccess) {
        bb_env_destroy(e);
        return fail(-2, "bb_env_create: cudaMemset state", err);
    }
    if ((err = cudaMalloc(&e->d_expand_scratch, (size_t)bb_expand_scratch_count(n_envs) * sizeof(int64_t))) != cudaSuccess) {
        bb_env_destroy(e);
        return fail(-2, "bb_env_create: cudaMalloc expand scratch", err);
    }
    // the first reset (the reference constructs each GameEngine with a dealt trio)
    err = bb_launch_reset(e->arr, nullptr, nullptr, 0);
    if (err == cudaSuccess) err = cudaDeviceSynchronize();
    if (err != cudaSuccess) {
        bb_env_destroy(e);
        return fail(-2, "bb_env_create: reset kernel", err);
    }
    *out = e;
    return 0;
}

int bb_env_destroy(bb_env* e) {
    if (!e) return 0;
    cudaFree(e->arr.s0); cudaFree(e->arr.s1); cudaFree(e->arr.s2);
    cudaFree(e->d_actions); cudaFree(e->d_block); cudaFree(e->d_dense); cudaFree(e->d_trios);
    cudaFree(e->d_expand_scratch);
    delete e;
    return 0;
}

int64_t bb_env_num_envs(const bb_env* e) { return e ? e->arr.n : -1; }

int bb_env_set_episode_end_buffer(bb_env* e, void* records) {
    if (!e) return fail(-1, "bb_env_set_episode_end_buffer: env is NULL");
    e->arr.ep_end = (BBEpisodeEnd*)records;
    return 0;
}

int bb_env_set_trios(bb_env* e, const uint8_t* h_trios, int64_t len, void* stream) {
    if (!e) return fail(-1, "bb_env_set_trios: env is NULL");
    BB_DEVICE(e, "bb_env_set_trios");
    cudaStream_t s = (cudaStream_t)stream;
    if (!h_trios) {                      // back to the Philox streams
        BB_CUDA(cudaStreamSynchronize(s), "bb_env_set_trios sync");
        cudaFree(e->d_trios);
        e->d_trios = nullptr; e->arr.trios = nullptr; e->arr.trio_len = 0;
        return 0;
    }
    if (len <= 0) return fail(-1, "bb_env_set_trios: len must be > 0");
    const size_t bytes = (size_t)e->arr.n * (size_t)len * 3;
    for (size_t k = 0; k < bytes; ++k)
        if (h_trios[k] >= BB_NUM_PIECES) return fail(-1, "bb_env_set_trios: piece index out of range");
    uint8_t* d = nullptr;
    BB_CUDA(cudaMalloc(&d, bytes), "bb_env_set_trios: cudaMalloc");
    cudaError_t err = cudaMemcpyAsync(d, h_trios, bytes, cudaMemcpyHostToDevice, s);
    if (err == cudaSuccess) err = cudaStreamSynchronize(s);
    if (err != cudaSuccess) { cudaFree(d); return fail(-2, "bb_env_set_trios: copy", err); }
    cudaFree(e->d_trios);
    e->d_trios = d; e->arr.trios = d; e->arr.trio_len = len;
    BB_CUDA(bb_launch_zero_draw_ctr(e->arr, s), "bb_env_set_trios: draw counters");
    return 0;
}

int bb_env_reset(bb_env* e, const uint8_t* reset_mask, uint64_t* mask_out, void* stream) {
    if (!e) return fail(-1, "bb_env_reset: env is NULL");
    BB_DEVICE(e, "bb_env_reset");
    BB_CUDA(bb_launch_reset(e->arr, reset_mask, mask_out, (cudaStream_t)stream), "bb_env_reset launch");
    return 0;
}

int bb_env_step(bb_env* e, const int32_t* actions, float* rewards, uint8_t* terminated,
                uint64_t* mask_out, uint64_t* board_out, uint32_t* pieces_out, int32_t* ep_score, int32_t* ep_len,
                uint32_t* info_out, uint64_t* stats, void* stream) {
    if (!e) return fail(-1, "bb_env_step: env is NULL");
    if (!actions || !rewards || !terminated) return fail(-1, "bb_env_step: actions/rewards/terminated are required");
    BB_DEVICE(e, "bb_env_step");
    BB_CUDA(bb_launch_step(e->arr, e->cfg, actions, rewards, terminated, mask_out, board_out, pieces_out, ep_score, ep_len,
                           info_out, (unsigned long long*)stats, (cudaStream_t)stream), "bb_env_step launch");
    return 0;
}

int bb_env_step_random(bb_env* e, int32_t n_steps, int32_t* actions_out, float* rewards, uint8_t* terminated,
                       uint64_t* mask_out, uint64_t* stats, const uint64_t* mask_in, void* stream) {
    if (!e) return fail(-1, "bb_env_step_random: env is NULL");
    if (n_steps < 1 || n_steps > (1 << 20)) return fail(-1, "bb_env_step_random: n_steps must be in [1, 2^20]");
    BB_DEVICE(e, "bb_env_step_random");
    BB_CUDA(bb_launch_step_random(e->arr, e->cfg, n_steps, 0, actions_out, rewards, terminated, mask_out,
                                  (unsigned long long*)stats, mask_in, (cudaStream_t)stream), "bb_env_step_random launch");
    return 0;
}

int bb_env_rollout_random(bb_env* e, int32_t n_steps, int32_t* actions_out, float* rewards, uint8_t* terminated,
                          uint64_t* mask_out, uint64_t* stats, void* stream) {
    if (!e) return fail(-1, "bb_env_rollout_random: env is NULL");
    if (n_steps < 1 || n_steps > (1 << 20)) return fail(-1, "bb_env_rollout_random: n_steps must be in [1, 2^20]");
    BB_DEVICE(e, "bb_env_rollout_random");
    BB_CUDA(bb_launch_step_random(e->arr, e->cfg, n_steps, 1, actions_out, rewards, terminated, mask_out,
                                  (unsigned long long*)stats, nullptr, (cudaStream_t)stream), "bb_env_rollout_random launch");
    return 0;
}

int bb_env_observe(bb_env* e, uint64_t* board_out, uint32_t* pieces_out, uint64_t* mask_out, void* stream) {
    if (!e) return fail(-1, "bb_env_observe: env is NULL");
    BB_DEVICE(e, "bb_env_observe");
    BB_CUDA(bb_launch_observe(e->arr, board_out, pieces_out, mask_out, (cudaStream_t)stream), "bb_env_observe launch");
    return 0;
}

int bb_env_sample_valid_actions(bb_env* e, uint64_t call_counter, int32_t* actions_out, int32_t* h_actions_out, void* stream) {
    if (!e) return fail(-1, "bb_env_sample_valid_actions: env is NULL");
    if (!actions_out && !h_actions_out) return fail(-1, "bb_env_sample_valid_actions: no output given");
    BB_DEVICE(e, "bb_env_sample_valid_actions");
    cudaStream_t s = (cudaStream_t)stream;
    int32_t* d = actions_out;
    if (!d) {
        if (int rc = ensure_staging(e)) return rc;
        d = e->d_actions;
    }
    BB_CUDA(bb_launch_sample_valid(e->arr, call_counter, d, s), "bb_env_sample_valid_actions launch");
    if (h_actions_out) {
        BB_CUDA(cudaMemcpyAsync(h_actions_out, d, e->arr.n * sizeof(int32_t), cudaMemcpyDeviceToHost, s), "D2H actions");
        BB_CUDA(cudaStreamSynchronize(s), "bb_env_sample_valid_actions sync");
    }
    return 0;
}

int bb_env_expand(bb_env* e, uint64_t call_counter, int32_t samples, int64_t capacity, int64_t* offsets,
                  int32_t* action_out, float* reward_out, uint8_t* terminated_out, uint32_t* info_out,
                  uint64_t* board_out, uint32_t* pieces_out, uint64_t* mask_out, void* stream) {
    if (!e) return fail(-1, "bb_env_expand: env is NULL");
    if (!offsets) return fail(-1, "bb_env_expand: offsets is NULL (it is always written)");
    if (samples < 1 || samples > 64) return fail(-1, "bb_env_expand: samples must be in [1, 64]");
    if (call_counter >= (1ull << 25)) return fail(-1, "bb_env_expand: call_counter must be < 2^25");
    if (capacity < 0) return fail(-1, "bb_env_expand: negative capacity");
    BB_DEVICE(e, "bb_env_expand");
    BB_CUDA(bb_launch_expand(e->arr, e->cfg, (uint32_t)call_counter, samples, capacity, offsets, e->d_expand_scratch,
                             action_out, reward_out, terminated_out, info_out, board_out, pieces_out, mask_out,
                             (cudaStream_t)stream), "bb_env_expand launch");
    return 0;
}

int bb_env_get_state(bb_env* e, void* host_records, void* stream) {
    if (!e || !host_records) return fail(-1, "bb_env_get_state: NULL argument");
    BB_DEVICE(e, "bb_env_get_state");
    const int64_t n = e->arr.n;
    uint4* tmp = (uint4*)malloc((size_t)n * 3 * sizeof(uint4));
    if (!tmp) return fail(-3, "bb_env_get_state: out of host memory");
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t err = cudaMemcpyAsync(tmp, e->arr.s0, n * sizeof(uint4), cudaMemcpyDeviceToHost, s);
    if (err == cudaSuccess) err = cudaMemcpyAsync(tmp + n, e->arr.s1, n * sizeof(uint4), cudaMemcpyDeviceToHost, s);
    if (err == cudaSuccess) err = cudaMemcpyAsync(tmp + 2 * n, e->arr.s2, n * sizeof(uint4), cudaMemcpyDeviceToHost, s);
    if (err == cudaSuccess) err = cudaStreamSynchronize(s);
    if (err != cudaSuccess) { free(tmp); return fail(-2, "bb_env_get_state copy", err); }
    uint4* rec = (uint4*)host_records;
    for (int64_t i = 0; i < n; ++i) { rec[3 * i] = tmp[i]; rec[3 * i + 1] = tmp[n + i]; rec[3 * i + 2] = tmp[2 * n + i]; }
    free(tmp);
    return 0;
}

int bb_env_set_state(bb_env* e, const void* host_records, void* stream) {
    if (!e || !host_records) return fail(-1, "bb_env_set_state: NULL argument");
    BB_DEVICE(e, "bb_env_set_state");
    const int64_t n = e->arr.n;
    uint4* tmp = (uint4*)malloc((size_t)n * 3 * sizeof(uint4));
    if (!tmp) return fail(-3, "bb_env_set_state: out of host memory");
    const uint4* rec = (const uint4*)host_records;
    for (int64_t i = 0; i < n; ++i) {
        const uint32_t p = rec[3 * i].z;
        if ((p & 0xFF) >= BB_NUM_PIECES || ((p >> 8) & 0xFF) >= BB_NUM_PIECES || ((p >> 16) & 0xFF) >= BB_NUM_PIECES) {
            free(tmp);
            return fail(-1, "bb_env_set_state: piece index out of range");
        }
        tmp[i] = rec[3 * i]; tmp[n + i] = rec[3 * i + 1]; tmp[2 * n + i] = rec[3 * i + 2];
    }
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t err = cudaMemcpyAsync(e->arr.s0, tmp, n * sizeof(uint4), cudaMemcpyHostToDevice, s);
    if (err == cudaSuccess) err = cudaMemcpyAsync(e->arr.s1, tmp + n, n * sizeof(uint4), cudaMemcpyHostToDevice, s);
    if (err == cudaSuccess) err = cudaMemcpyAsync(e->arr.s2, tmp + 2 * n, n * sizeof(uint4), cudaMemcpyHostToDevice, s);
    if (err == cudaSuccess) err = cudaStreamSynchronize(s);
    free(tmp);
    if (err != cudaSuccess) return fail(-2, "bb_env_set_state copy", err);
    return 0;
}

// Result arrays of the host-buffer step, as byte offsets into ONE block of `total` bytes:
// [0] mask u64[3][n], [1] board u64[n], [2] rewards f32[n], [3] pieces u32[n], [7] terminated u8[n] form
// the PREFIX (41 B/env, rounded up to 16) every step needs; [4] ep_score i32[n], [5] ep_len i32[n],
// [6] info u32[n] follow it.  A caller whose host arrays sit in one pinned block at these offsets gets
// the prefix (or, when it also passes the three tail arrays, the whole block) in ONE device-to-host
// copy; the tail of the last step can be fetched later with bb_env_fetch_step_info.
int bb_env_host_layout(int64_t n_envs, int64_t offsets8[8], int64_t* total_bytes, int64_t* prefix_bytes) {
    if (n_envs <= 0 || !offsets8 || !total_bytes) return fail(-1, "bb_env_host_layout: bad argument");
    const int64_t n = n_envs;
    const int64_t prefix = (41 * n + 15) / 16 * 16;
    offsets8[0] = 0; offsets8[1] = 24 * n; offsets8[2] = 32 * n; offsets8[3] = 36 * n; offsets8[7] = 40 * n;
    offsets8[4] = prefix; offsets8[5] = prefix + 4 * n; offsets8[6] = prefix + 8 * n;
    *total_bytes = prefix + 12 * n;
    if (prefix_bytes) *prefix_bytes = prefix;
    return 0;
}

static int ensure_staging(bb_env* e) {
    if (e->d_block) return 0;
    const int64_t n = e->arr.n;
    int64_t off[8], total;
    bb_env_host_layout(n, off, &total, nullptr);
    int32_t* da = nullptr;
    uint8_t* db = nullptr;
    cudaError_t err = cudaMalloc(&da, n * sizeof(int32_t));
    if (err == cudaSuccess) err = cudaMalloc(&db, (size_t)total);
    if (err == cudaSuccess) err = cudaMemset(db, 0, (size_t)total);
    if (err != cudaSuccess) {
        cudaFree(da); cudaFree(db);
        return fail(-2, "bb_env_step_host: staging buffers", err);
    }
    e->d_actions = da;
    e->d_block = db;
    e->d_mask = (uint64_t*)(e->d_block + off[0]);
    e->d_board = (uint64_t*)(e->d_block + off[1]);
    e->d_rewards = (float*)(e->d_block + off[2]);
    e->d_pieces = (uint32_t*)(e->d_block + off[3]);
    e->d_ep_score = (int32_t*)(e->d_block + off[4]);
    e->d_ep_len = (int32_t*)(e->d_block + off[5]);
    e->d_info = (uint32_t*)(e->d_block + off[6]);
    e->d_terminated = e->d_block + off[7];
    return 0;
}

int bb_env_step_host(bb_env* e, const int32_t* h_actions, float* h_rewards, uint8_t* h_terminated,
                     uint64_t* h_board, uint32_t* h_pieces, uint64_t* h_mask, int32_t* h_ep_score,
                     int32_t* h_ep_len, uint32_t* h_info, void* stream) {
    if (!e) return fail(-1, "bb_env_step_host: env is NULL");
    if (!h_actions || !h_rewards || !h_terminated) return fail(-1, "bb_env_step_host: actions/rewards/terminated are required");
    BB_DEVICE(e, "bb_env_step_host");
    if (int rc = ensure_staging(e)) return rc;
    const int64_t n = e->arr.n;
    cudaStream_t s = (cudaStream_t)stream;
    BB_CUDA(cudaMemcpyAsync(e->d_actions, h_actions, n * sizeof(int32_t), cudaMemcpyHostToDevice, s), "H2D actions");
    // the step kernel writes the packed next observation (board, pieces) itself; the per-step info
    // arrays always land in the device staging block (bb_env_fetch_step_info reads them later)
    BB_CUDA(bb_launch_step_range(e->arr, e->cfg, 0, n, e->d_actions, e->d_rewards, e->d_terminated,
                                 e->d_mask, e->d_ep_score, e->d_ep_len, e->d_info, e->d_board, e->d_pieces, s),
            "bb_env_step_host launch");
    int64_t off[8], total, prefix;
    bb_env_host_layout(n, off, &total, &prefix);
    uint8_t* hb = (uint8_t*)h_mask;
    const bool prefix_block = hb && (uint8_t*)h_board == hb + off[1] && (uint8_t*)h_rewards == hb + off[2] &&
                              (uint8_t*)h_pieces == hb + off[3] && h_terminated == hb + off[7];
    const bool tail_block = (uint8_t*)h_ep_score == hb + off[4] && (uint8_t*)h_ep_len == hb + off[5] &&
                            (uint8_t*)h_info == hb + off[6];
    const bool no_tail = !h_ep_score && !h_ep_len && !h_info;
    if (prefix_block && (tail_block || no_tail)) {
        // one transfer (41 B/env, or 53 B/env with the info tail) instead of up to eight calls, each of
        // which costs several microseconds of driver time
        BB_CUDA(cudaMemcpyAsync(hb, e->d_block, (size_t)(tail_block ? total : 41 * n), cudaMemcpyDeviceToHost, s), "D2H results");
    } else {
        BB_CUDA(cudaMemcpyAsync(h_rewards, e->d_rewards, n * sizeof(float), cudaMemcpyDeviceToHost, s), "D2H rewards");
        BB_CUDA(cudaMemcpyAsync(h_terminated, e->d_terminated, n, cudaMemcpyDeviceToHost, s), "D2H terminated");
        if (h_board) BB_CUDA(cudaMemcpyAsync(h_board, e->d_board, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, s), "D2H board");
        if (h_pieces) BB_CUDA(cudaMemcpyAsync(h_pieces, e->d_pieces, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, s), "D2H pieces");
        if (h_mask) BB_CUDA(cudaMemcpyAsync(h_mask, e->d_mask, 3 * n * sizeof(uint64_t), cudaMemcpyDeviceToHost, s), "D2H mask");
        if (h_ep_score) BB_CUDA(cudaMemcpyAsync(h_ep_score, e->d_ep_score, n * sizeof(int32_t), cudaMemcpyDeviceToHost, s), "D2H ep_score");
        if (h_ep_len) BB_CUDA(cudaMemcpyAsync(h_ep_len, e->d_ep_len, n * sizeof(int32_t), cudaMemcpyDeviceToHost, s), "D2H ep_len");
        if (h_info) BB_CUDA(cudaMemcpyAsync(h_info, e->d_info, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, s), "D2H info");
    }
    BB_CUDA(cudaStreamSynchronize(s), "bb_env_step_host sync");
    return 0;
}

int bb_env_fetch_step_info(bb_env* e, int32_t* h_ep_score, int32_t* h_ep_len, uint32_t* h_info, void* stream) {
    if (!e) return fail(-1, "bb_env_fetch_step_info: env is NULL");
    BB_DEVICE(e, "bb_env_fetch_step_info");
    if (!e->d_block) return fail(-1, "bb_env_fetch_step_info: no host-buffer step has run yet");
    const int64_t n = e->arr.n;
    cudaStream_t s = (cudaStream_t)stream;
    if (h_ep_score && h_ep_len && h_info && (uint8_t*)h_ep_len == (uint8_t*)h_ep_score + 4 * n &&
        (uint8_t*)h_info == (uint8_t*)h_ep_score + 8 * n) {
        BB_CUDA(cudaMemcpyAsync(h_ep_score, e->d_ep_score, 12 * n, cudaMemcpyDeviceToHost, s), "D2H step info");
    } else {
        if (h_ep_score) BB_CUDA(cudaMemcpyAsync(h_ep_score, e->d_ep_score, n * sizeof(int32_t), cudaMemcpyDeviceToHost, s), "D2H ep_score");
        if (h_ep_len) BB_CUDA(cudaMemcpyAsync(h_ep_len, e->d_ep_len, n * sizeof(int32_t), cudaMemcpyDeviceToHost, s), "D2H ep_len");
        if (h_info) BB_CUDA(cudaMemcpyAsync(h_info, e->d_info, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, s), "D2H info");
    }
    BB_CUDA(cudaStreamSynchronize(s), "bb_env_fetch_step_info sync");
    return 0;
}

// Reference-layout ("dense") result block: [0] board f32[n][8][8], [1] pieces f32[n][3][8][8],
// [2] action_mask i8[n][192], [3] rewards f32[n], [4] terminated u8[n]  = 1,221 B/env.
int bb_env_host_dense_layout(int64_t n_envs, int64_t offsets5[5], int64_t* total_bytes) {
    if (n_envs <= 0 || !offsets5 || !total_bytes) return fail(-1, "bb_env_host_dense_layout: bad argument");
    const int64_t n = n_envs;
    offsets5[0] = 0; offsets5[1] = 256 * n; offsets5[2] = 1024 * n; offsets5[3] = 1216 * n; offsets5[4] = 1220 * n;
    *total_bytes = 1221 * n;
    return 0;
}

static int ensure_dense(bb_env* e) {
    if (e->d_dense) return 0;
    int64_t off[5], total;
    bb_env_host_dense_layout(e->arr.n, off, &total);
    uint8_t* d = nullptr;
    cudaError_t err = cudaMalloc(&d, (size_t)total);
    if (err == cudaSuccess) err = cudaMemset(d, 0, (size_t)total);
    if (err != cudaSuccess) { cudaFree(d); return fail(-2, "bb_env_step_host_dense: staging buffer", err); }
    e->d_dense = d;
    return 0;
}

// expand the packed observation in the staging block into the dense block and bring it to the host
static int dense_to_host(bb_env* e, void* h_block, cudaStream_t s) {
    const int64_t n = e->arr.n;
    int64_t off[5], total;
    bb_env_host_dense_layout(n, off, &total);
    BB_CUDA(bb_launch_unpack_obs(e->d_board, e->d_pieces, e->d_mask, n, e->d_dense + off[0], BB_F32, e->d_dense + off[2],
                                 BB_U8, n, s, e->d_dense + off[1]), "dense observation expand");
    BB_CUDA(cudaMemcpyAsync(h_block, e->d_dense, (size_t)total, cudaMemcpyDeviceToHost, s), "D2H dense results");
    BB_CUDA(cudaStreamSynchronize(s), "dense results sync");
    return 0;
}

int bb_env_step_host_dense(bb_env* e, const int32_t* h_actions, void* h_block, void* stream) {
    if (!e) return fail(-1, "bb_env_step_host_dense: env is NULL");
    if (!h_actions || !h_block) return fail(-1, "bb_env_step_host_dense: actions and the result block are required");
    BB_DEVICE(e, "bb_env_step_host_dense");
    if (int rc = ensure_staging(e)) return rc;
    if (int rc = ensure_dense(e)) return rc;
    const int64_t n = e->arr.n;
    int64_t off[5], total;
    bb_env_host_dense_layout(n, off, &total);
    cudaStream_t s = (cudaStream_t)stream;
    BB_CUDA(cudaMemcpyAsync(e->d_actions, h_actions, n * sizeof(int32_t), cudaMemcpyHostToDevice, s), "H2D actions");
    // rewards / terminated go straight into the dense block, the packed observation into the staging block
    BB_CUDA(bb_launch_step_range(e->arr, e->cfg, 0, n, e->d_actions, (float*)(e->d_dense + off[3]), e->d_dense + off[4],
                                 e->d_mask, e->d_ep_score, e->d_ep_len, e->d_info, e->d_board, e->d_pieces, s),
            "bb_env_step_host_dense launch");
    return dense_to_host(e, h_block, s);
}

int bb_env_observe_host_dense(bb_env* e, void* h_block, void* stream) {
    if (!e) return fail(-1, "bb_env_observe_host_dense: env is NULL");
    if (!h_block) return fail(-1, "bb_env_observe_host_dense: the result block is required");
    BB_DEVICE(e, "bb_env_observe_host_dense");
    if (int rc = ensure_staging(e)) return rc;
    if (int rc = ensure_dense(e)) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    BB_CUDA(bb_launch_observe(e->arr, e->d_board, e->d_pieces, e->d_mask, s), "bb_env_observe_host_dense launch");
    return dense_to_host(e, h_block, s);
}

int bb_unpack_obs(const uint64_t* board, const uint32_t* pieces, const uint64_t* mask, int64_t mask_stride,
                  void* obs_nchw, int obs_dtype, void* mask_dense, int mask_dtype, int64_t n, void* stream) {
    if (n < 0) return fail(-1, "bb_unpack_obs: negative n");
    if (obs_nchw && obs_dtype != BB_F32 && obs_dtype != BB_BF16) return fail(-1, "bb_unpack_obs: obs_dtype must be BB_F32 or BB_BF16");
    if (mask_dense && mask_dtype != BB_F32 && mask_dtype != BB_U8) return fail(-1, "bb_unpack_obs: mask_dtype must be BB_F32 or BB_U8");
    if (n == 0) return 0;
    if (obs_nchw && (!board || !pieces)) return fail(-1, "bb_unpack_obs: board/pieces required for obs");
    if (mask_dense && !mask) return fail(-1, "bb_unpack_obs: mask required for mask_dense");
    BB_CUDA(bb_launch_unpack_obs(board, pieces, mask, mask_stride, obs_nchw, obs_dtype, mask_dense, mask_dtype, n,
                                 (cudaStream_t)stream), "bb_unpack_obs launch");
    return 0;
}

int bb_unpack_obs_reference_layout(const uint64_t* board, const uint32_t* pieces, const uint64_t* mask, int64_t mask_stride,
                                   float* board_f32, float* pieces_f32, int8_t* action_mask_i8, int64_t n, void* stream) {
    if (n < 0) return fail(-1, "bb_unpack_obs_reference_layout: negative n");
    if (n == 0) return 0;
    if (!board || !pieces || !board_f32 || !pieces_f32) return fail(-1, "bb_unpack_obs_reference_layout: board/pieces arrays are required");
    if (action_mask_i8 && !mask) return fail(-1, "bb_unpack_obs_reference_layout: mask required for action_mask");
    BB_CUDA(bb_launch_unpack_obs(board, pieces, mask, mask_stride, board_f32, BB_F32, action_mask_i8, BB_U8, n,
                                 (cudaStream_t)stream, pieces_f32), "bb_unpack_obs_reference_layout launch");
    return 0;
}

int bb_gather_minibatch(const int64_t* index, int64_t batch, int64_t n_envs, const uint64_t* board, const uint32_t* pieces,
                        const uint64_t* mask, const int32_t* action, const float* logp, const float* adv, const float* ret,
                        const float* adv_mean_std, void* obs_nchw, int obs_dtype, uint64_t* mask_out, int32_t* action_out,
                        float* logp_out, float* adv_out, float* ret_out, void* stream) {
    if (batch < 0 || n_envs <= 0) return fail(-1, "bb_gather_minibatch: bad size");
    if (obs_nchw && obs_dtype != BB_F32 && obs_dtype != BB_BF16)
        return fail(-1, "bb_gather_minibatch: obs_dtype must be BB_F32 or BB_BF16");
    if (batch == 0) return 0;
    // obs_nchw == NULL: no observation planes (the symmetric update expands eight views with bb_unpack_obs_sym)
    if (!index || !board || !pieces || !mask || !action || !logp || !adv || !ret || !mask_out || !action_out ||
        !logp_out || !adv_out || !ret_out)
        return fail(-1, "bb_gather_minibatch: NULL array");
    BB_CUDA(bb_launch_gather_minibatch(index, batch, n_envs, board, pieces, mask, action, logp, adv, ret, adv_mean_std,
                                       obs_nchw, obs_dtype, mask_out, action_out, logp_out, adv_out, ret_out,
                                       (cudaStream_t)stream), "bb_gather_minibatch launch");
    return 0;
}

int bb_unpack_obs_sym(const uint64_t* board, const uint32_t* pieces, const int64_t* index, void* obs_nchw, int obs_dtype,
                      int64_t n, void* stream) {
    if (n < 0) return fail(-1, "bb_unpack_obs_sym: negative n");
    if (obs_dtype != BB_F32 && obs_dtype != BB_BF16) return fail(-1, "bb_unpack_obs_sym: obs_dtype must be BB_F32 or BB_BF16");
    if (n == 0) return 0;
    if (!board || !pieces || !obs_nchw) return fail(-1, "bb_unpack_obs_sym: board/pieces/obs_nchw are required");
    BB_CUDA(bb_launch_unpack_obs_sym(board, pieces, index, obs_nchw, obs_dtype, n, (cudaStream_t)stream),
            "bb_unpack_obs_sym launch");
    return 0;
}

int bb_sym_logits_mean(const void* logits, int logits_dtype, const uint32_t* pieces, float* out, int64_t n, void* stream) {
    if (n < 0) return fail(-1, "bb_sym_logits_mean: negative n");
    if (logits_dtype != BB_F32 && logits_dtype != BB_BF16) return fail(-1, "bb_sym_logits_mean: logits_dtype must be BB_F32 or BB_BF16");
    if (n == 0) return 0;
    if (!logits || !pieces || !out) return fail(-1, "bb_sym_logits_mean: NULL array");
    if ((uintptr_t)logits & 15) return fail(-1, "bb_sym_logits_mean: logits must be 16-byte aligned");
    BB_CUDA(bb_launch_sym_logits_mean(logits, logits_dtype, pieces, out, n, (cudaStream_t)stream), "bb_sym_logits_mean launch");
    return 0;
}

int bb_sym_logits_mean_backward(const float* grad_out, const uint32_t* pieces, void* grad_logits, int logits_dtype, int64_t n,
                                void* stream) {
    if (n < 0) return fail(-1, "bb_sym_logits_mean_backward: negative n");
    if (logits_dtype != BB_F32 && logits_dtype != BB_BF16)
        return fail(-1, "bb_sym_logits_mean_backward: logits_dtype must be BB_F32 or BB_BF16");
    if (n == 0) return 0;
    if (!grad_out || !pieces || !grad_logits) return fail(-1, "bb_sym_logits_mean_backward: NULL array");
    if ((uintptr_t)grad_logits & 15) return fail(-1, "bb_sym_logits_mean_backward: grad_logits must be 16-byte aligned");
    BB_CUDA(bb_launch_sym_logits_mean_bwd(grad_out, pieces, grad_logits, logits_dtype, n, (cudaStream_t)stream),
            "bb_sym_logits_mean_backward launch");
    return 0;
}

int bb_sym_canonical(const uint64_t* board, const uint32_t* pieces, const int64_t* index, uint64_t* board_out,
                     uint32_t* pieces_out, uint8_t* views_out, int64_t n, void* stream) {
    if (n < 0) return fail(-1, "bb_sym_canonical: negative n");
    if (n == 0) return 0;
    if (!board || !pieces || !board_out || !pieces_out || !views_out) return fail(-1, "bb_sym_canonical: NULL array");
    BB_CUDA(bb_launch_sym_canonical(board, pieces, index, board_out, pieces_out, views_out, n, (cudaStream_t)stream),
            "bb_sym_canonical launch");
    return 0;
}

int bb_sym_logits_canonical(const void* logits, int logits_dtype, const uint32_t* pieces, const uint8_t* views, float* out,
                            int64_t n, void* stream) {
    if (n < 0) return fail(-1, "bb_sym_logits_canonical: negative n");
    if (logits_dtype != BB_F32 && logits_dtype != BB_BF16)
        return fail(-1, "bb_sym_logits_canonical: logits_dtype must be BB_F32 or BB_BF16");
    if (n == 0) return 0;
    if (!logits || !pieces || !views || !out) return fail(-1, "bb_sym_logits_canonical: NULL array");
    if ((uintptr_t)logits & 15) return fail(-1, "bb_sym_logits_canonical: logits must be 16-byte aligned");
    BB_CUDA(bb_launch_sym_logits_canonical(logits, logits_dtype, pieces, views, out, n, (cudaStream_t)stream),
            "bb_sym_logits_canonical launch");
    return 0;
}

int bb_sym_logits_canonical_backward(const float* grad_out, const uint32_t* pieces, const uint8_t* views, void* grad_logits,
                                     int logits_dtype, int64_t n, void* stream) {
    if (n < 0) return fail(-1, "bb_sym_logits_canonical_backward: negative n");
    if (logits_dtype != BB_F32 && logits_dtype != BB_BF16)
        return fail(-1, "bb_sym_logits_canonical_backward: logits_dtype must be BB_F32 or BB_BF16");
    if (n == 0) return 0;
    if (!grad_out || !pieces || !views || !grad_logits) return fail(-1, "bb_sym_logits_canonical_backward: NULL array");
    if (((uintptr_t)grad_out | (uintptr_t)grad_logits) & 15)
        return fail(-1, "bb_sym_logits_canonical_backward: grad_out and grad_logits must be 16-byte aligned");
    BB_CUDA(bb_launch_sym_logits_canonical_bwd(grad_out, pieces, views, grad_logits, logits_dtype, n, (cudaStream_t)stream),
            "bb_sym_logits_canonical_backward launch");
    return 0;
}

int bb_masked_sample(const void* logits, int logits_dtype, const uint64_t* mask, int64_t mask_stride,
                     uint64_t seed, uint64_t call_counter, int mode, int32_t* action, float* logp,
                     float* entropy, int64_t n, int64_t row_offset, const uint64_t* call_counter_dev, void* stream) {
    if (n < 0) return fail(-1, "bb_masked_sample: negative n");
    if (logits_dtype != BB_F32 && logits_dtype != BB_BF16) return fail(-1, "bb_masked_sample: logits_dtype must be BB_F32 or BB_BF16");
    if (mode < 0 || mode > 2) return fail(-1, "bb_masked_sample: mode must be 0, 1 or 2");
    if (n == 0) return 0;
    if (!logits || !mask || !action) return fail(-1, "bb_masked_sample: logits/mask/action are required");
    BB_CUDA(bb_launch_masked_sample(logits, logits_dtype, mask, mask_stride, seed, call_counter, mode, action, logp,
                                    entropy, n, (cudaStream_t)stream, row_offset, call_counter_dev), "bb_masked_sample launch");
    return 0;
}

int bb_masked_head_backward(const void* logits, int logits_dtype, const uint64_t* mask, int64_t mask_stride,
                            const int32_t* action, const float* grad_logp, const float* grad_entropy,
                            void* grad_logits, int64_t n, void* stream) {
    if (n < 0) return fail(-1, "bb_masked_head_backward: negative n");
    if (logits_dtype != BB_F32 && logits_dtype != BB_BF16) return fail(-1, "bb_masked_head_backward: logits_dtype must be BB_F32 or BB_BF16");
    if (n == 0) return 0;
    if (!logits || !mask || !action || !grad_logp || !grad_logits) return fail(-1, "bb_masked_head_backward: NULL array");
    BB_CUDA(bb_launch_masked_head_bwd(logits, logits_dtype, mask, mask_stride, action, grad_logp, grad_entropy, grad_logits,
                                      n, (cudaStream_t)stream), "bb_masked_head_backward launch");
    return 0;
}

int bb_ppo_loss(const void* logits, int logits_dtype, const uint64_t* mask, int64_t mask_stride,
                const int32_t* action, const float* old_logp, const float* advantages, const float* returns,
                const float* values, double clip_epsilon, double value_coef, double entropy_coef,
                void* grad_logits, float* grad_values, double* sums5, int64_t n, void* stream) {
    if (n < 0) return fail(-1, "bb_ppo_loss: negative n");
    if (logits_dtype != BB_F32 && logits_dtype != BB_BF16) return fail(-1, "bb_ppo_loss: logits_dtype must be BB_F32 or BB_BF16");
    if (n == 0) return 0;
    if (!logits || !mask || !action || !old_logp || !advantages || !returns || !values || !grad_logits || !grad_values || !sums5)
        return fail(-1, "bb_ppo_loss: NULL array");
    BB_CUDA(bb_launch_ppo_loss(logits, logits_dtype, mask, mask_stride, action, old_logp, advantages, returns, values,
                               (float)clip_epsilon, (float)value_coef, (float)entropy_coef, grad_logits, grad_values,
                               sums5, n, (cudaStream_t)stream), "bb_ppo_loss launch");
    return 0;
}

int64_t bb_bn_workspace_size(int channels) {
    if (channels <= 0 || channels % 8 != 0 || channels > 2048) return -1;
    return (int64_t)bb_bn_workspace_floats(channels);
}

static int bn_check(int64_t rows, int channels) {
    if (rows < 0) return fail(-1, "bb_bn_relu: negative rows");
    if (channels <= 0 || channels % 8 != 0 || channels > 2048) return fail(-1, "bb_bn_relu: channels must be a multiple of 8 in [8, 2048]");
    return 0;
}

int bb_bn_relu_forward(const void* x, const void* skip, const float* gamma, const float* beta, const float* pre_bias,
                       float* running_mean,
                       float* running_var, double momentum, double eps, int training, void* y, float* save_mean,
                       float* save_rstd, float* workspace, int64_t rows, int channels, void* stream) {
    if (bn_check(rows, channels)) return -1;
    if (rows == 0) return 0;
    if (!x || !gamma || !beta || !y || !workspace) return fail(-1, "bb_bn_relu_forward: NULL array");
    if (training && (!save_mean || !save_rstd)) return fail(-1, "bb_bn_relu_forward: training needs save_mean / save_rstd");
    if (!training && (!running_mean || !running_var)) return fail(-1, "bb_bn_relu_forward: eval needs the running statistics");
    BB_CUDA(bb_launch_bn_relu_fwd(x, skip, gamma, beta, pre_bias, running_mean, running_var, (float)momentum, (float)eps, training, y,
                                  save_mean, save_rstd, workspace, rows, channels, (cudaStream_t)stream), "bb_bn_relu_forward launch");
    return 0;
}

int bb_bn_relu_backward(const void* x, const void* y, const void* grad_y, const float* gamma, const float* save_mean,
                        const float* save_rstd, void* grad_x, void* grad_skip, float* grad_gamma, float* grad_beta,
                        float* workspace, int64_t rows, int channels, void* stream) {
    if (bn_check(rows, channels)) return -1;
    if (rows == 0) return 0;
    if (!x || !y || !grad_y || !gamma || !save_mean || !save_rstd || !grad_x || !grad_gamma || !grad_beta || !workspace)
        return fail(-1, "bb_bn_relu_backward: NULL array");
    BB_CUDA(bb_launch_bn_relu_bwd(x, y, grad_y, gamma, save_mean, save_rstd, grad_x, grad_skip, grad_gamma, grad_beta, workspace,
                                  rows, channels, (cudaStream_t)stream), "bb_bn_relu_backward launch");
    return 0;
}

int bb_bn_relu_backward_no_skip(const void* x, const void* grad_y, const float* gamma, const float* beta,
                                const float* save_mean, const float* save_rstd, void* grad_x, float* grad_gamma,
                                float* grad_beta, float* workspace, int64_t rows, int channels, void* stream) {
    if (bn_check(rows, channels)) return -1;
    if (rows == 0) return 0;
    if (!x || !grad_y || !gamma || !beta || !save_mean || !save_rstd || !grad_x || !grad_gamma || !grad_beta || !workspace)
        return fail(-1, "bb_bn_relu_backward_no_skip: NULL array");
    BB_CUDA(bb_launch_bn_relu_bwd(x, nullptr, grad_y, gamma, save_mean, save_rstd, grad_x, nullptr, grad_gamma, grad_beta, workspace,
                                  rows, channels, (cudaStream_t)stream, beta), "bb_bn_relu_backward_no_skip launch");
    return 0;
}

int bb_gae(const float* rewards, const float* values, const float* dones, const float* last_values,
           double gamma, double lam, float* adv, float* ret, double* moments, int64_t T, int64_t N, void* stream) {
    if (T < 0 || N < 0) return fail(-1, "bb_gae: negative size");
    if (T == 0 || N == 0) return 0;                 // empty rollout: nothing to do (pointers may be NULL)
    if (!rewards || !values || !dones || !last_values || !adv || !ret) return fail(-1, "bb_gae: NULL array");
    // numpy casts the Python doubles gamma and gamma*lambda to float32 before the array multiply
    BB_CUDA(bb_launch_gae(rewards, values, dones, last_values, (float)gamma, (float)(gamma * lam), adv, ret, moments,
                          T, N, (cudaStream_t)stream), "bb_gae launch");
    return 0;
}

}  // extern "C"
