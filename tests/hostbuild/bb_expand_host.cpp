// Host (g++) build of the one-ply expansion (bb_env_expand) on top of the product's rules header
// csrc/bb_rules.cuh — TEST INFRASTRUCTURE, the expansion counterpart of bb_rules_host.cpp.  The same
// per-item code the sm_100a kernel runs (bb_expand_count / bb_expand_item / bb_env_pre / bb_env_post),
// with the sequential bb_deal on the LOOKAHEAD source, so it can be checked against the oracle without a
// GPU and the GPU kernel can be checked against it.  The product never loads this library.
#include "bb_rules.cuh"
#include <string.h>

static BBTables g_tables;
static bool g_init = false;
static void init() { if (!g_init) { bb_fill_tables(&g_tables); g_init = true; } }

extern "C" {

int64_t bbx_state_size() { return (int64_t)sizeof(BBState); }

// bb_env_expand with the sequential deal on the LOOKAHEAD source: same item order and outputs
// (mask plane-major with plane stride `capacity`); states are not modified
void bbx_expand(const BBState* s, int64_t n, const double cfg[7], uint64_t seed, int64_t env_offset,
                uint32_t call_counter, int samples, int64_t capacity, int64_t* offsets, int32_t* action_out,
                float* reward_out, uint8_t* terminated_out, uint32_t* info_out, uint64_t* board_out,
                uint32_t* pieces_out, uint64_t* mask_out) {
    init();
    BBRewardCfg c;
    memcpy(&c, cfg, sizeof(c));
    BBLookaheadSrc src;
    src.seed = seed; src.call_counter = call_counter;
    int64_t item = 0;
    for (int64_t i = 0; i < n; ++i) {
        offsets[i] = item;
        uint64_t m[3];
        bb_action_mask(s[i], &g_tables, m);
        const int cnt = bb_expand_count(s[i], m, samples);
        const uint64_t env_id = (uint64_t)(env_offset + i);
        for (int j = 0; j < cnt; ++j, ++item) {
            if (item >= capacity) continue;
            int k;
            const int a = bb_expand_item(s[i], m, samples, j, &k);
            BBState t = s[i];
            BBStepOut o;
            const BBMove mv = bb_env_pre(t, a, &g_tables, o);
            uint32_t draws = 0;
            if (mv.needs_deal) {
                uint32_t d = (uint32_t)k << 8;
                t.pieces = bb_deal(t.board, &g_tables, src, env_id, &d);
                draws = d - ((uint32_t)k << 8);
            }
            bb_env_post(t, mv, draws, &g_tables, c, BBTrioSrc(seed), env_id, BB_FLAG_NO_AUTO_RESET, o);
            if (action_out) action_out[item] = a;
            if (reward_out) reward_out[item] = o.reward;
            if (terminated_out) terminated_out[item] = (uint8_t)o.terminated;
            if (info_out) info_out[item] = o.info;
            if (board_out) board_out[item] = t.board;
            if (pieces_out) pieces_out[item] = t.pieces;
            if (mask_out) for (int p = 0; p < 3; ++p) mask_out[p * capacity + item] = o.mask[p];
        }
    }
    offsets[n] = item;
}
uint32_t bbx_lookahead_trio(uint64_t seed, uint64_t env_id, uint32_t call_counter, uint32_t k, uint32_t d) {
    BBLookaheadSrc src;
    src.seed = seed; src.call_counter = call_counter;
    return bb_candidate(src, env_id, (k << 8) | d);
}

}  // extern "C"
