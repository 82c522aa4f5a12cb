// Host (g++) build of the board-symmetry functions of the product's rules header csrc/bb_rules.cuh —
// TEST INFRASTRUCTURE, the symmetry counterpart of bb_rules_host.cpp.  It exposes bb_sym_* and one env
// step on an injected candidate-trio stream (bb_env_apply), so that the symmetry tables, the group laws
// and the equivariance of the rules can be checked against the oracle without a GPU, and the eight-view
// kernels against it on the GPU.  The product never loads this library.
#include "bb_rules.cuh"
#include <string.h>

static BBTables g_tables;
static BBSymTables g_sym;
static bool g_init = false;
static void init() { if (!g_init) { bb_fill_tables(&g_tables); bb_fill_sym_tables(&g_sym); g_init = true; } }

extern "C" {

int64_t bbs_state_size() { return (int64_t)sizeof(BBState); }

void bbs_tables(uint8_t* perm /* [8][40] */, uint8_t* shift /* [8][40] */) {
    init();
    memcpy(perm, g_sym.perm, sizeof(g_sym.perm));
    memcpy(shift, g_sym.shift, sizeof(g_sym.shift));
}
uint64_t bbs_sym_board(int g, uint64_t b) { return bb_sym_board(g, b); }
int bbs_sym_cell(int g, int a) { return bb_sym_cell(g, a); }
uint32_t bbs_sym_pieces(int g, uint32_t pw) { init(); return bb_sym_pieces(&g_sym, g, pw); }
int bbs_sym_anchor(int g, uint32_t id, int a) { init(); return bb_sym_anchor(&g_sym, g, id, a); }
uint64_t bbs_sym_mask_plane(int g, uint32_t id, uint64_t plane) { init(); return bb_sym_mask_plane(&g_sym, g, id, plane); }

// view g of packed rows: out[(g*n + i)*4 + k] = bitboard of plane k (board, then the three piece planes,
// 0 for a used slot or an id >= 37), the planes the eight-view observation kernel writes
void bbs_obs_views(const uint64_t* board, const uint32_t* pieces, int64_t n, uint64_t* out) {
    init();
    for (int g = 0; g < BB_SYM_N; ++g)
        for (int64_t i = 0; i < n; ++i) {
            uint64_t* o = out + ((int64_t)g * n + i) * 4;
            const uint32_t pw = bb_sym_pieces(&g_sym, g, pieces[i]);
            o[0] = bb_sym_board(g, board[i]);
            for (int k = 0; k < 3; ++k) {
                const uint32_t id = (pw >> (8 * k)) & 0xFFu;
                o[1 + k] = ((pw >> (24 + k)) & 1u) || id >= BB_NUM_PIECES ? 0ull : BB_HOST_PIECE_MASKS[id];
            }
        }
}

// per-row symmetry g[i]: transformed packed rows, mask planes [3][n] (pieces = the ORIGINAL rows' words; a
// slot whose id is >= 37 gives 0) and actions
void bbs_sym_rows(const int32_t* g, const uint64_t* board, const uint32_t* pieces, int64_t n, uint64_t* board_out,
                  uint32_t* pieces_out) {
    init();
    for (int64_t i = 0; i < n; ++i) {
        board_out[i] = bb_sym_board(g[i], board[i]);
        pieces_out[i] = bb_sym_pieces(&g_sym, g[i], pieces[i]);
    }
}
void bbs_sym_mask_rows(const int32_t* g, const uint32_t* pieces, const uint64_t* mask, int64_t n, uint64_t* out) {
    init();
    for (int k = 0; k < 3; ++k)
        for (int64_t i = 0; i < n; ++i) {
            const uint32_t id = (pieces[i] >> (8 * k)) & 0xFFu;
            out[k * n + i] = id < BB_NUM_PIECES ? bb_sym_mask_plane(&g_sym, g[i], id, mask[k * n + i]) : 0ull;
        }
}
void bbs_sym_action_rows(const int32_t* g, const uint32_t* pieces, const int32_t* action, int64_t n, int32_t* out) {
    init();
    for (int64_t i = 0; i < n; ++i) {
        const int s = action[i] >> 6;
        const uint32_t id = (pieces[i] >> (8 * s)) & 0xFFu;
        out[i] = s * 64 + bb_sym_anchor(&g_sym, g[i], id, action[i] & 63);
    }
}

// one step of state *s on the injected candidate trios[len][3] (draws wrap), no auto-reset
void bbs_step(BBState* s, int action, const double cfg[7], const uint8_t* trios, int64_t len, float* reward,
              uint8_t* terminated, uint32_t* info, uint64_t mask[3]) {
    init();
    BBRewardCfg c;
    memcpy(&c, cfg, sizeof(c));
    BBTrioSrc src(0);
    src.trios = trios; src.len = len; src.base = 0;
    BBStepOut o;
    bb_env_apply(*s, action, &g_tables, c, src, 0, BB_FLAG_NO_AUTO_RESET, o);
    *reward = o.reward;
    *terminated = (uint8_t)o.terminated;
    *info = o.info;
    mask[0] = o.mask[0]; mask[1] = o.mask[1]; mask[2] = o.mask[2];
}

}  // extern "C"
