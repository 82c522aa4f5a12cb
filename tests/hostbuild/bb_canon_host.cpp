// Host (g++) build of the canonical-view function of the product's rules header csrc/bb_rules.cuh (bb_sym_canonical)
// — TEST INFRASTRUCTURE, the canonical-frame counterpart of bb_sym_host.cpp.  It lets the definition of the
// canonical view and its view set be checked against a numpy restatement without a GPU, and the device kernel
// against it on the GPU.  The product never loads this library.
#include "bb_rules.cuh"

static BBSymTables g_sym;
static bool g_init = false;

extern "C" {

// canonical view (board_out, pieces_out) and view set (views) of each packed row
void bbc_canonical(const uint64_t* board, const uint32_t* pieces, int64_t n, uint64_t* board_out, uint32_t* pieces_out,
                   uint8_t* views) {
    if (!g_init) { bb_fill_sym_tables(&g_sym); g_init = true; }
    for (int64_t i = 0; i < n; ++i) views[i] = (uint8_t)bb_sym_canonical(&g_sym, board[i], pieces[i], board_out + i, pieces_out + i);
}

}  // extern "C"
