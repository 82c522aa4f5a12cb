// bb_rules.cuh — Block Blast rules on 64-bit bitboards, shared by the sm_100a kernels and by
// a host (g++) build used only to fuzz this file against the oracle without a GPU.
//
// Bit convention: bit = row*8 + col (same as the action codec a % 64,
// reference src/environment/block_blast_env.py:114-118).  A piece is its cell mask with the
// top-left of its bounding box at bit 0, the mask of anchors that keep it on the board, and
// the list of its cell offsets.
//
// What each function restates (file:line in the reference):
//   bb_valid        Board.can_place for all 64 anchors at once     src/game/board.py:71-93, :117-142
//   bb_clear        find_complete_lines + clear_lines              src/game/board.py:144-193
//   bb_holes        Board.count_holes                              src/game/board.py:195-216
//   bb_center       filled cells of rows/cols 2..5                 src/game/board.py:236-243
//   bb_classify /   _can_place_all_pieces (a boolean, so the       src/game/engine.py:174-238
//   bb_branch       search order is free)
//   bb_env_pre      BlockBlastEnv.step validation + make_move up   block_blast_env.py:224-245,
//                   to the trio regeneration                       engine.py:390-437
//   bb_env_post     game over, reward, auto-reset, next mask       engine.py:440-441, block_blast_env.py:148-193,
//                                                                  src/environment/wrappers.py:96-102
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define BB_HD __host__ __device__ __forceinline__
#else
#define BB_HD inline
#endif

#include "bb_piece_table.inc"
#include "bb_sym_table.inc"

// ---------------------------------------------------------------------------------------
// tables
// ---------------------------------------------------------------------------------------
#define BB_TABLE_N (BB_NUM_PIECES + 3)
// one 32-byte row per piece (rows 37..39 are zero padding), so a piece is two 16-byte fetches
struct alignas(16) BBTableRow {
    uint64_t mask;   // piece cells at the origin
    uint64_t inb;    // anchors whose bounding box stays on the board
    uint64_t offs;   // valid-mask recipe, one byte each: a0..a3, b1, b2 (see bb_valid)
    uint32_t meta;   // n | h<<4 | w<<8 | maxrow<<12 | maxcol<<16
    uint32_t pad;
};
struct BBTables { BBTableRow row[BB_TABLE_N]; };

#define BB_META_N(m) ((m) & 0xFu)
#define BB_META_MAXROW(m) (((m) >> 12) & 0xFu)
#define BB_META_MAXCOL(m) (((m) >> 16) & 0xFu)

static const uint64_t BB_HOST_PIECE_MASKS[BB_NUM_PIECES] = BB_PIECE_MASKS;
static const uint64_t BB_HOST_PIECE_INB[BB_NUM_PIECES] = BB_PIECE_INB;
static const uint64_t BB_HOST_PIECE_OFFS[BB_NUM_PIECES] = BB_PIECE_OFFS;
static const uint32_t BB_HOST_PIECE_META[BB_NUM_PIECES] = BB_PIECE_META;

inline void bb_fill_tables(BBTables* t) {
    for (int i = 0; i < BB_TABLE_N; ++i) {
        t->row[i].mask = i < BB_NUM_PIECES ? BB_HOST_PIECE_MASKS[i] : 0;
        t->row[i].inb = i < BB_NUM_PIECES ? BB_HOST_PIECE_INB[i] : 0;
        t->row[i].offs = i < BB_NUM_PIECES ? BB_HOST_PIECE_OFFS[i] : 0;
        t->row[i].meta = i < BB_NUM_PIECES ? BB_HOST_PIECE_META[i] : 0;
        t->row[i].pad = 0;
    }
}

struct BBPiece { uint64_t pm, inb, offs; uint32_t meta; };

BB_HD BBPiece bb_piece(const BBTables* T, uint32_t id) {
    BBPiece p;
#if defined(__CUDA_ARCH__)
    const uint4* r = reinterpret_cast<const uint4*>(&T->row[id]);
    const uint4 a = r[0], b = r[1];
    p.pm = (uint64_t)a.x | ((uint64_t)a.y << 32);
    p.inb = (uint64_t)a.z | ((uint64_t)a.w << 32);
    p.offs = (uint64_t)b.x | ((uint64_t)b.y << 32);
    p.meta = b.z;
#else
    p.pm = T->row[id].mask; p.inb = T->row[id].inb; p.offs = T->row[id].offs; p.meta = T->row[id].meta;
#endif
    return p;
}

// ---------------------------------------------------------------------------------------
// bit helpers
// ---------------------------------------------------------------------------------------
BB_HD int bb_popc(uint64_t x) {
#if defined(__CUDA_ARCH__)
    return __popcll(x);
#else
    return __builtin_popcountll(x);
#endif
}
BB_HD int bb_popc32(uint32_t x) {
#if defined(__CUDA_ARCH__)
    return __popc(x);
#else
    return __builtin_popcount(x);
#endif
}
BB_HD int bb_ctz(uint64_t x) {   // x != 0
#if defined(__CUDA_ARCH__)
    const uint32_t lo = (uint32_t)x;
    return lo ? (__ffs((int)lo) - 1) : (31 + __ffs((int)(uint32_t)(x >> 32)));
#else
    return __builtin_ctzll(x);
#endif
}
BB_HD uint32_t bb_mulhi(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}
// position of the k-th (0-based) set bit of w; k < popcount(w).  Binary search on popcounts.
BB_HD int bb_select(uint64_t w, int k) {
#if defined(__CUDA_ARCH__)
    uint32_t x = (uint32_t)w;
    int pos = 0;
    int c = __popc(x);
    if (k >= c) { k -= c; pos = 32; x = (uint32_t)(w >> 32); }
    c = __popc(x & 0xFFFFu);
    if (k >= c) { k -= c; pos += 16; x >>= 16; }
    c = __popc(x & 0xFFu);
    if (k >= c) { k -= c; pos += 8; x >>= 8; }
    c = __popc(x & 0xFu);
    if (k >= c) { k -= c; pos += 4; x >>= 4; }
    c = __popc(x & 0x3u);
    if (k >= c) { k -= c; pos += 2; x >>= 2; }
    if (k >= (int)(x & 1u)) pos += 1;
    return pos;
#else
    for (int i = 0; i < k; ++i) w &= w - 1;
    return __builtin_ctzll(w);
#endif
}

#define BB_COL_A 0x0101010101010101ull
#define BB_COL_H 0x8080808080808080ull
#define BB_CENTER 0x00003C3C3C3C0000ull

// ---------------------------------------------------------------------------------------
// board primitives
// ---------------------------------------------------------------------------------------
// e >> o for 0 <= o <= 32
BB_HD uint64_t bb_shr(uint64_t e, uint32_t o) {
#if defined(__CUDA_ARCH__)
    const uint32_t lo = (uint32_t)e, hi = (uint32_t)(e >> 32);
    return (uint64_t)__funnelshift_rc(lo, hi, o) | ((uint64_t)__funnelshift_rc(hi, 0u, o) << 32);
#else
    return e >> o;
#endif
}

// byte k (0..3) of a 32-bit word, zero-extended: one PRMT on the device
BB_HD uint32_t bb_byte(uint32_t w, int k) {
#if defined(__CUDA_ARCH__)
    return __byte_perm(w, 0u, 0x4440u + (uint32_t)k);
#else
    return (w >> (8 * k)) & 0xFFu;
#endif
}

// All anchors at which piece p fits on the EMPTY-cell set e = ~board: board.py:71-93 for the
// 64 anchors at once.  Every piece is a Minkowski sum  A (+) {0,b1} (+) {0,b2}  of a base shape
// of at most four cells and two doubling steps (tools/gen_piece_tables.py: the 3x3 square is
// (0,1,2) (+) {0,8} (+) {0,8}; pieces of up to four cells have b1 = b2 = 0), so the mask is four
// shift-ANDs of e and two shift-ANDs of the intermediate result — the same six steps for all 37
// pieces, no branch on the piece size.  Anchors whose bounding box leaves the board are removed
// by the in-bounds mask at the end (a shifted-in or wrapped cell can only belong to those).
BB_HD uint64_t bb_valid(uint64_t e, const BBPiece& p) {
    const uint32_t lo = (uint32_t)p.offs, hi = (uint32_t)(p.offs >> 32);
    uint64_t v = bb_shr(e, bb_byte(lo, 0)) & bb_shr(e, bb_byte(lo, 1));
    v &= bb_shr(e, bb_byte(lo, 2)) & bb_shr(e, lo >> 24);
    v &= bb_shr(v, bb_byte(hi, 0));
    v &= bb_shr(v, bb_byte(hi, 1));
    return v & p.inb;
}

// Rows of a 32-bit half board (one byte per row).  A byte is 0xFF iff adding 1 to its low seven
// bits carries into bit 7 while bit 7 is set; the sum cannot carry into the next byte.
// bb_rowflags32: bit 7 of byte r = row r full (other bits unspecified);
// bb_rowmask32: 0xFF in every full row's byte, 0 elsewhere (sign-replicating PRMT on the device).
BB_HD uint32_t bb_rowflags32(uint32_t x) { return ((x & 0x7F7F7F7Fu) + 0x01010101u) & x; }
BB_HD uint32_t bb_rowmask32(uint32_t x) {
#if defined(__CUDA_ARCH__)
    uint32_t m;   // selector nibbles 8..B: replicate the sign bit of byte 0..3 (__byte_perm cannot)
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(m) : "r"(bb_rowflags32(x)), "r"(0u), "r"(0xBA98u));
    return m;
#else
    return ((bb_rowflags32(x) & 0x80808080u) >> 7) * 0xFFu;
#endif
}
// bit c set iff column c is full
BB_HD uint32_t bb_fullcols(uint32_t lo, uint32_t hi) {
    uint32_t c = lo & hi;
    c &= c >> 16;
    c &= c >> 8;
    return c & 0xFFu;
}

// Full rows / columns are detected on the same board, then all removed (board.py:166-193).
// Returns the cleared board; *lines = rows + cols.
BB_HD uint64_t bb_clear(uint64_t b, int* lines) {
    const uint32_t lo = (uint32_t)b, hi = (uint32_t)(b >> 32);
    const uint32_t rl = bb_rowmask32(lo), rh = bb_rowmask32(hi), c = bb_fullcols(lo, hi);
    const uint32_t cm = c * 0x01010101u;
    *lines = ((bb_popc32(rl) + bb_popc32(rh)) >> 3) + bb_popc32(c);
    return (uint64_t)(lo & ~(rl | cm)) | ((uint64_t)(hi & ~(rh | cm)) << 32);
}

// true iff b has at least one full row or column
BB_HD bool bb_any_full(uint64_t b) {
    const uint32_t lo = (uint32_t)b, hi = (uint32_t)(b >> 32);
    return ((((bb_rowflags32(lo) | bb_rowflags32(hi)) & 0x80808080u) | bb_fullcols(lo, hi))) != 0u;
}

BB_HD uint64_t bb_clear_only(uint64_t b) {
    int l;
    return bb_clear(b, &l);
}

// b with its full rows/columns removed; *full tells whether there were any (one pass)
BB_HD uint64_t bb_clear_if_full(uint64_t b, bool* full) {
    const uint32_t lo = (uint32_t)b, hi = (uint32_t)(b >> 32);
    const uint32_t rl = bb_rowmask32(lo), rh = bb_rowmask32(hi), c = bb_fullcols(lo, hi);
    const uint32_t cm = c * 0x01010101u;
    *full = (rl | rh | c) != 0u;
    return (uint64_t)(lo & ~(rl | cm)) | ((uint64_t)(hi & ~(rh | cm)) << 32);
}

// board.py:195-216: empty cells whose four neighbours are filled or off-board.
BB_HD int bb_holes(uint64_t b) {
    const uint64_t up = (b << 8) | 0xFFull;                      // neighbour in row-1 (row 0: off-board)
    const uint64_t dn = (b >> 8) | 0xFF00000000000000ull;        // neighbour in row+1
    const uint64_t lf = ((b << 1) & ~BB_COL_A) | BB_COL_A;       // neighbour in col-1
    const uint64_t rt = ((b >> 1) & ~BB_COL_H) | BB_COL_H;       // neighbour in col+1
    return bb_popc(~b & up & dn & lf & rt);
}

BB_HD int bb_center(uint64_t b) { return bb_popc(b & BB_CENTER); }

// Line occupancy summary of a board: byte r of `rows` = filled cells of row r (0..8); `colp` =
// the filled-cell counts of the eight columns in BIT-SLICED form: byte j holds, for every column
// c (bit c), bit j of that column's count (a carry-save adder tree over the eight row bytes: 17
// logic ops for all columns at once).  Used for "which lines can a piece complete" bounds.
struct BBLines { uint64_t rows; uint32_t colp; };

BB_HD uint32_t bb_maj(uint32_t x, uint32_t y, uint32_t z) { return (x & y) | (x & z) | (y & z); }

BB_HD BBLines bb_lines(uint64_t b) {
    BBLines L;
    uint64_t t = b - ((b >> 1) & 0x5555555555555555ull);
    t = (t & 0x3333333333333333ull) + ((t >> 2) & 0x3333333333333333ull);
    L.rows = (t + (t >> 4)) & 0x0F0F0F0F0F0F0F0Full;
    const uint32_t lo = (uint32_t)b, hi = (uint32_t)(b >> 32);
    // rows k and k+4 -> 2-bit counts per byte lane
    const uint32_t a1 = lo ^ hi, b1 = lo & hi;
    // byte lanes k and k+2 -> 3-bit counts in lanes 0, 1
    const uint32_t c = a1 & (a1 >> 16);
    const uint32_t a2 = a1 ^ (a1 >> 16), b2 = b1 ^ (b1 >> 16) ^ c, d2 = bb_maj(b1, b1 >> 16, c);
    // lanes 0 and 1 -> 4-bit counts in the low byte
    const uint32_t c1 = a2 & (a2 >> 8);
    const uint32_t ones = a2 ^ (a2 >> 8), twos = b2 ^ (b2 >> 8) ^ c1, c2 = bb_maj(b2, b2 >> 8, c1);
    const uint32_t fours = d2 ^ (d2 >> 8) ^ c2, eights = bb_maj(d2, d2 >> 8, c2);
    L.colp = (ones & 0xFFu) | ((twos & 0xFFu) << 8) | ((fours & 0xFFu) << 16) | ((eights & 0xFFu) << 24);
    return L;
}
// rows with at most m empty cells, as a byte mask (0xFF per such row), 1 <= m <= 7
BB_HD uint64_t bb_rows_within_mask(const BBLines& L, int m) {
    const uint64_t f = L.rows + (uint64_t)(0x78 + m) * BB_COL_A;   // bit 7 of a byte: count + 120 + m >= 128
#if defined(__CUDA_ARCH__)
    uint32_t lo, hi;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(lo) : "r"((uint32_t)f), "r"(0u), "r"(0xBA98u));
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(hi) : "r"((uint32_t)(f >> 32)), "r"(0u), "r"(0xBA98u));
    return (uint64_t)lo | ((uint64_t)hi << 32);
#else
    return ((f & BB_COL_H) >> 7) * 0xFFull;
#endif
}
// columns with at most m empty cells, as an 8-bit column mask: count + m >= 8 by a ripple carry
// over the bit-sliced counts (1 <= m <= 7)
BB_HD uint32_t bb_cols_within_bits(const BBLines& L, int m) {
    const uint32_t ones = L.colp & 0xFFu, twos = (L.colp >> 8) & 0xFFu, fours = (L.colp >> 16) & 0xFFu, eights = L.colp >> 24;
    const uint32_t m0 = 0u - ((uint32_t)m & 1u), m1 = 0u - (((uint32_t)m >> 1) & 1u), m2 = 0u - (((uint32_t)m >> 2) & 1u);
    const uint32_t k0 = ones & m0;
    const uint32_t k1 = bb_maj(twos, m1, k0);
    const uint32_t k2 = bb_maj(fours, m2, k1);
    return (eights | k2) & 0xFFu;
}
// exists a row with at most m empty cells / a column with at most m empty cells (1 <= m <= 7)
BB_HD bool bb_row_within(const BBLines& L, int m) {
    return ((L.rows + (uint64_t)(0x78 + m) * BB_COL_A) & BB_COL_H) != 0;   // count + 120 + m >= 128
}
BB_HD bool bb_col_within(const BBLines& L, int m) { return bb_cols_within_bits(L, m) != 0u; }

// Anchors of piece p whose placement covers at least one cell of T (the OR twin of bb_valid:
// same recipe, OR instead of AND).  A superset is fine for its users, so wrapped bits are not
// filtered here; the valid mask they are combined with removes out-of-bounds anchors.
BB_HD uint64_t bb_cover(uint64_t T, const BBPiece& p) {
    const uint32_t lo = (uint32_t)p.offs, hi = (uint32_t)(p.offs >> 32);
    uint64_t v = bb_shr(T, bb_byte(lo, 0)) | bb_shr(T, bb_byte(lo, 1));
    v |= bb_shr(T, bb_byte(lo, 2)) | bb_shr(T, lo >> 24);
    v |= bb_shr(v, bb_byte(hi, 0));
    v |= bb_shr(v, bb_byte(hi, 1));
    return v;
}

// Anchors (a superset of those) at which placing p on board bb can complete a line: a completed
// line has at most maxrow(p) (row) / maxcol(p) (column) empty cells and p covers all of them, in
// particular one of them — so the anchor lies in the cover of the empty cells of such lines.
BB_HD uint64_t bb_clearing_candidates(uint64_t bb, const BBLines& L, const BBPiece& p) {
    const uint64_t near = bb_rows_within_mask(L, (int)BB_META_MAXROW(p.meta)) |
                          ((uint64_t)bb_cols_within_bits(L, (int)BB_META_MAXCOL(p.meta)) * BB_COL_A);
    return bb_cover(~bb & near, p);
}

// ---------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. SC'11).  Stream layout documented in philox.py.
// ---------------------------------------------------------------------------------------
struct BBPhilox4 { uint32_t x, y, z, w; };

BB_HD BBPhilox4 bb_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi0 = bb_mulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = bb_mulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    BBPhilox4 r = {c0, c1, c2, c3};
    return r;
}

#define BB_STREAM_TRIO 0u
#define BB_STREAM_POLICY 1u
#define BB_STREAM_SAMPLE 2u

// candidate trio number `draw` of global env `env_id`: three ids in [0,37), packed in bytes 0..2
BB_HD uint32_t bb_draw_trio(uint64_t seed, uint64_t env_id, uint32_t draw) {
    const BBPhilox4 r = bb_philox((uint32_t)env_id, (uint32_t)(env_id >> 32), draw, BB_STREAM_TRIO,
                                  (uint32_t)seed, (uint32_t)(seed >> 32));
    return bb_mulhi(r.x, 37u) | (bb_mulhi(r.y, 37u) << 8) | (bb_mulhi(r.z, 37u) << 16);
}

// Where candidate trios come from.  Product runs: Philox stream (seed, global env id, draw).
// Replay / parity runs (bb_env_set_trios): an injected table trios[n][len][3] of piece ids — what
// the reference's engine.rng.choice(37, size=3) (src/game/pieces.py:350-355) returned, draw by
// draw — so the reference's own numpy-PCG64 games can be replayed on the GPU.  Row = env id - base;
// draws past the table wrap around.  Implicitly constructible from a seed (= Philox).
struct BBTrioSrc {
    uint64_t seed;
    const uint8_t* trios;
    int64_t len, base;
    BB_HD BBTrioSrc(uint64_t s = 0) : seed(s), trios(nullptr), len(0), base(0) {}
};

BB_HD uint32_t bb_candidate(const BBTrioSrc& src, uint64_t env_id, uint32_t draw) {
    if (src.trios) {
        const uint8_t* t = src.trios + (((int64_t)env_id - src.base) * src.len + (int64_t)(draw % (uint32_t)src.len)) * 3;
        return (uint32_t)t[0] | ((uint32_t)t[1] << 8) | ((uint32_t)t[2] << 16);
    }
    return bb_draw_trio(src.seed, env_id, draw);
}

// LOOKAHEAD stream (bb_env_expand): the trio dealt to a SUCCESSOR state that placed the env's last
// unused piece.  Independent of the env's own TRIO stream, so a planner never reads the deck it
// will be dealt from.  Sample k of call `call_counter`, candidate d (0..99) of that deal:
//   counter = (env_id lo, env_id hi, call_counter << 7 | d, 4 | k << 8)   (call_counter < 2^25, k < 64)
// The deal loops pass `draw` = k << 8 | d (the k of the item travels with the draw counter, which the
// warp deal shuffles from the owner lane), so the source itself holds only what the warp shares.
#define BB_STREAM_LOOKAHEAD 4u
struct BBLookaheadSrc {
    uint64_t seed;
    uint32_t call_counter;
};

BB_HD uint32_t bb_candidate(const BBLookaheadSrc& src, uint64_t env_id, uint32_t draw) {
    const BBPhilox4 r = bb_philox((uint32_t)env_id, (uint32_t)(env_id >> 32), (src.call_counter << 7) | (draw & 0xFFu),
                                  BB_STREAM_LOOKAHEAD | (draw >> 8 << 8), (uint32_t)src.seed, (uint32_t)(src.seed >> 32));
    return bb_mulhi(r.x, 37u) | (bb_mulhi(r.y, 37u) << 8) | (bb_mulhi(r.z, 37u) << 16);
}

// ---------------------------------------------------------------------------------------
// trio solvability (engine.py:174-238).  The reference enumerates piece orders and anchors
// depth-first with line clears after every simulated placement and returns a boolean, so any
// sound and complete search gives the identical result.  Facts used:
//   (M) clearing lines only removes cells, so a placement that fits before a clear fits after.
//   (P) hence if the three pieces have pairwise-disjoint placements that all fit on the
//       current board, every order works ("packing"), no simulation needed;
//   (C) conversely a solution that is NOT a packing must complete a line with its first or
//       second placement; a line with `miss` empty cells can only be completed by pieces that
//       can put at least `miss` cells into one row (column): meta maxrow / maxcol.
// The search is cut into independent BRANCHES (one first-level placement each) so that the
// kernel can spread one hard (board, trio) item over a team of lanes:
//   stage A branch t < nA : x at its t-th anchor, then a packing of y and z beside it
//   stage B branch        : piece i at one of its anchors (any order i), then the other two
//                           with clears simulated; when nothing cleared, only a CLEARING
//                           second placement is explored (a plain packing is stage A's job)
// ---------------------------------------------------------------------------------------
#ifdef BB_COUNT_WORK
struct BBWork { long long valid_calls, fast_accept, fast_reject, pack_iters, clear_iters, slow, branches; };
static BBWork g_bb_work;
#define BB_WORK(f, n) (g_bb_work.f += (n))
#else
#define BB_WORK(f, n) ((void)0)
#endif

enum { BB_REJECT = 0, BB_ACCEPT = 1, BB_HARD = 2 };

struct BBItem {
    uint64_t b;        // board the trio must be placeable on
    uint64_t v[3];     // valid anchors of each piece on b
    uint32_t plan;     // bits 0-1 x, 2-3 y, 4-5 z (stage-A order); bits 8-15 nA; bits 16-23 nB
};
#define BB_PLAN_NA(p) (((p) >> 8) & 0xFFu)
#define BB_PLAN_NB(p) (((p) >> 16) & 0xFFu)

// piece i of three without dynamic indexing (keeps everything in registers on the device)
BB_HD BBPiece bb_pick3(const BBPiece& p0, const BBPiece& p1, const BBPiece& p2, int i) {
    BBPiece r;
    r.pm = i == 0 ? p0.pm : (i == 1 ? p1.pm : p2.pm);
    r.inb = i == 0 ? p0.inb : (i == 1 ? p1.inb : p2.inb);
    r.offs = i == 0 ? p0.offs : (i == 1 ? p1.offs : p2.offs);
    r.meta = i == 0 ? p0.meta : (i == 1 ? p1.meta : p2.meta);
    return r;
}

// fact (C) for three pieces: can the two largest per-line contributions complete any line?
BB_HD bool bb_clear_reachable(uint64_t b, const BBPiece& p0, const BBPiece& p1, const BBPiece& p2) {
    const int r0 = (int)BB_META_MAXROW(p0.meta), r1 = (int)BB_META_MAXROW(p1.meta), r2 = (int)BB_META_MAXROW(p2.meta);
    const int c0 = (int)BB_META_MAXCOL(p0.meta), c1 = (int)BB_META_MAXCOL(p1.meta), c2 = (int)BB_META_MAXCOL(p2.meta);
    const int rmin = r0 < r1 ? (r0 < r2 ? r0 : r2) : (r1 < r2 ? r1 : r2);
    const int cmin = c0 < c1 ? (c0 < c2 ? c0 : c2) : (c1 < c2 ? c1 : c2);
    const int rt = r0 + r1 + r2 - rmin, ct = c0 + c1 + c2 - cmin;
    if (rt >= 8 || ct >= 8) return true;      // two pieces could even fill an empty line
    const BBLines L = bb_lines(b);
    return bb_row_within(L, rt) || bb_col_within(L, ct);
}

// Cheap classification of (board, trio): ACCEPT / REJECT when provable with a handful of
// valid-mask evaluations, else HARD with the item's branch plan filled in.
BB_HD int bb_classify(uint64_t b, const BBPiece& p0, const BBPiece& p1, const BBPiece& p2, BBItem* it) {
    const uint64_t e = ~b;
    it->b = b;
    it->v[0] = bb_valid(e, p0);
    it->v[1] = bb_valid(e, p1);
    it->v[2] = bb_valid(e, p2);
    BB_WORK(valid_calls, 3);
    const int n0 = bb_popc(it->v[0]), n1 = bb_popc(it->v[1]), n2 = bb_popc(it->v[2]);
    uint32_t nA = 0, order = 0;
    if (n0 && n1 && n2) {
        // greedy packing: fewest anchors first, lowest anchors
        int x = 0, y = 1, z = 2;
        if (n1 < n0 && n1 <= n2) { x = 1; y = 0; }
        else if (n2 < n0 && n2 < n1) { x = 2; z = 0; }
        const int ny = (y == 0 ? n0 : (y == 1 ? n1 : n2)), nz = (z == 0 ? n0 : (z == 1 ? n1 : n2));
        if (nz < ny) { const int s_ = y; y = z; z = s_; }
        const BBPiece px = bb_pick3(p0, p1, p2, x), py = bb_pick3(p0, p1, p2, y), pz = bb_pick3(p0, p1, p2, z);
        const uint64_t vx = x == 0 ? it->v[0] : (x == 1 ? it->v[1] : it->v[2]);
        const uint64_t b1 = b | (px.pm << bb_ctz(vx));
        const uint64_t vy = bb_valid(~b1, py);
        BB_WORK(valid_calls, 1);
        if (vy) {
            // lowest and highest anchor of y: two cheap tries
            BB_WORK(valid_calls, 1);
            if (bb_valid(~(b1 | (py.pm << bb_ctz(vy))), pz)) return BB_ACCEPT;
            const int ah = 63 - (int)
#if defined(__CUDA_ARCH__)
                __clzll((long long)vy);
#else
                __builtin_clzll(vy);
#endif
            BB_WORK(valid_calls, 1);
            if (bb_valid(~(b1 | (py.pm << ah)), pz)) return BB_ACCEPT;
        }
        nA = (uint32_t)(x == 0 ? n0 : (x == 1 ? n1 : n2));
        order = (uint32_t)x | ((uint32_t)y << 2) | ((uint32_t)z << 4);
    }
    // stage B is only worth exploring if some line can be completed at all (fact C)
    const uint32_t nB = bb_clear_reachable(b, p0, p1, p2) ? (uint32_t)(n0 + n1 + n2) : 0u;
    it->plan = order | (nA << 8) | (nB << 16);
    if (nA + nB == 0) return BB_REJECT;
    return BB_HARD;
}

// A branch = one first-level placement already applied (board bb, cleared if it completed a
// line) plus up to two second-level scans, processed one anchor ("unit") at a time:
//   phase 0: piece A at each anchor of m0, then piece B must fit
//   phase 1: piece B at each anchor of m1, then piece A must fit
// A phase in "always" mode tests the leaf for every anchor; otherwise only for anchors whose
// placement completes a line (the no-clear case is covered elsewhere: fact P).
struct BBBranch {
    uint64_t bb, m0, m1;
    BBPiece A, B;
    uint32_t always;   // bit 0: phase 0 always, bit 1: phase 1 always, bit 2: roles of A and B swapped
};

BB_HD bool bb_can_complete_line(const BBLines& L, const BBPiece& p) {
    return bb_row_within(L, (int)BB_META_MAXROW(p.meta)) || bb_col_within(L, (int)BB_META_MAXCOL(p.meta));
}

#define BB_TRIO_ID(trio, i) (((trio) >> (8 * (i))) & 0xFFu)

// "Always" phase shortcut: one placement of A overlaps at most n(A) * n(B) anchors of B, so when B
// has more anchors than that, B fits beside ANY placement of A (a clear only makes more room):
// one anchor of A is enough, its unit proves solvability.  This removes the long loops after a
// clear has emptied the board (both pieces then have dozens of anchors).
BB_HD uint64_t bb_one_anchor_if_roomy(uint64_t mA, uint64_t vB, const BBPiece& A, const BBPiece& B) {
    const int roomy = bb_popc(vB) > (int)(BB_META_N(A.meta) * BB_META_N(B.meta));
    return roomy ? (mA & (0ull - mA)) : mA;
}

// open branch t of a HARD item, t in [0, nA + nB); pieces are fetched by role from the table
BB_HD void bb_branch_open(BBBranch& br, const BBItem& it, const BBTables* T, uint32_t trio, uint32_t t) {
    BB_WORK(branches, 1);
    const uint32_t nA = BB_PLAN_NA(it.plan);
    if (t < nA) {
        const int x = (int)(it.plan & 3u), y = (int)((it.plan >> 2) & 3u), z = (int)((it.plan >> 4) & 3u);
        const uint64_t vx = x == 0 ? it.v[0] : (x == 1 ? it.v[1] : it.v[2]);
        const uint64_t pmx = T->row[BB_TRIO_ID(trio, x)].mask;
        bool full;
        br.bb = bb_clear_if_full(it.b | (pmx << bb_select(vx, (int)t)), &full);
        br.A = bb_piece(T, BB_TRIO_ID(trio, y));
        br.B = bb_piece(T, BB_TRIO_ID(trio, z));
        BB_WORK(valid_calls, 2);
        // z must still fit beside x at all, else no packing goes through this anchor
        const uint64_t vA = bb_valid(~br.bb, br.A), vB = bb_valid(~br.bb, br.B);
        // walk the piece with fewer anchors (roles are symmetric for a packing), one anchor of it
        // when the other piece has more anchors than one placement can block
        const bool flip = bb_popc(vB) < bb_popc(vA);
        const uint64_t vf = flip ? vB : vA, vs = flip ? vA : vB;
        br.m0 = vs ? bb_one_anchor_if_roomy(vf, vs, br.A, br.B) : 0ull;
        br.m1 = 0ull;
        br.always = 1u | (flip ? 4u : 0u);
        return;
    }
    int k = (int)(t - nA);
    int i = 0;
    const int n0 = bb_popc(it.v[0]), n1 = bb_popc(it.v[1]);
    if (k >= n0) { k -= n0; i = 1; if (k >= n1) { k -= n1; i = 2; } }
    const int j = i == 0 ? 1 : 0, l = i == 2 ? 1 : 2;
    const uint64_t vi = i == 0 ? it.v[0] : (i == 1 ? it.v[1] : it.v[2]);
    const uint64_t pmi = T->row[BB_TRIO_ID(trio, i)].mask;
    bool full1;
    br.bb = bb_clear_if_full(it.b | (pmi << bb_select(vi, k)), &full1);
    br.A = bb_piece(T, BB_TRIO_ID(trio, j));
    br.B = bb_piece(T, BB_TRIO_ID(trio, l));
    const BBLines L = bb_lines(br.bb);
    BB_WORK(valid_calls, 2);
    // second placements that cannot complete a line are dropped here (they used to be tested one
    // by one in the unit loop): 4.2 -> 1.6 units per branch on boards from play
    const uint64_t vA = bb_valid(~br.bb, br.A), vB = bb_valid(~br.bb, br.B);
    const uint64_t cA = vA & bb_clearing_candidates(br.bb, L, br.A), cB = vB & bb_clearing_candidates(br.bb, L, br.B);
    // first placement cleared a line: everything about the two other pieces is open — walk all
    // anchors of one of them (the one with fewer; this covers the packings of both orders), the
    // other one first only where it clears itself.  Nothing cleared: a packing beside i is stage
    // A's business, only clearing second placements matter.
    const bool flip = full1 && bb_popc(vB) < bb_popc(vA);
    br.m0 = full1 ? bb_one_anchor_if_roomy(flip ? vB : vA, flip ? vA : vB, br.A, br.B) : cA;
    br.m1 = flip ? cA : cB;
    br.always = (full1 ? 1u : 0u) | (flip ? 4u : 0u);
}

// process one unit of an open branch (precondition: (m0 | m1) != 0); true = trio solvable
BB_HD bool bb_branch_unit(BBBranch& br) {
    const bool ph = br.m0 == 0ull;
    uint64_t m = ph ? br.m1 : br.m0;
    const int a = bb_ctz(m);
    m &= m - 1;
    if (ph) br.m1 = m; else br.m0 = m;
    // phase 0 places A and tests B, phase 1 the other way round; bit 2 of `always` swaps the roles
    const bool useB = ph != (((br.always >> 2) & 1u) != 0u);
    bool full;
    const uint64_t b2 = bb_clear_if_full(br.bb | ((useB ? br.B.pm : br.A.pm) << a), &full);
    BB_WORK(clear_iters, 1);
    if (!full && !((br.always >> (ph ? 1 : 0)) & 1u)) return false;
    BB_WORK(valid_calls, 1);
    BBPiece s2;
    s2.pm = 0;
    s2.inb = useB ? br.A.inb : br.B.inb;
    s2.offs = useB ? br.A.offs : br.B.offs;
    s2.meta = useB ? br.A.meta : br.B.meta;
    return bb_valid(~b2, s2) != 0ull;
}

// sequential drivers (host build): same branches and units, in index order
BB_HD bool bb_branch(const BBItem& it, const BBTables* T, uint32_t trio, uint32_t t) {
    BBBranch br;
    bb_branch_open(br, it, T, trio, t);
    while (br.m0 | br.m1)
        if (bb_branch_unit(br)) return true;
    return false;
}

BB_HD bool bb_solvable(uint64_t b, const BBTables* T, uint32_t trio) {
    BBPiece P[3];
    P[0] = bb_piece(T, trio & 0xFFu);
    P[1] = bb_piece(T, (trio >> 8) & 0xFFu);
    P[2] = bb_piece(T, (trio >> 16) & 0xFFu);
    BBItem it;
    const int f = bb_classify(b, P[0], P[1], P[2], &it);
    if (f == BB_ACCEPT) { BB_WORK(fast_accept, 1); return true; }
    if (f == BB_REJECT) { BB_WORK(fast_reject, 1); return false; }
    BB_WORK(slow, 1);
    const uint32_t n = BB_PLAN_NA(it.plan) + BB_PLAN_NB(it.plan);
    for (uint32_t t = 0; t < n; ++t)
        if (bb_branch(it, T, trio, t)) return true;
    return false;
}

// ---------------------------------------------------------------------------------------
// per-env state: 48 bytes = three 16-byte words (SoA of uint4 in HBM)
// ---------------------------------------------------------------------------------------
struct BBState {
    uint64_t board;
    uint32_t pieces;       // bytes 0..2 piece ids, byte 3 = used bits (bit i = piece i used)
    uint32_t aux;          // byte 0 prev_holes, byte 1 prev center filled count, byte 2 game over
    int32_t score, streak, moves, lines_total;
    int32_t max_streak, blocks_total;
    uint32_t draw_ctr;     // candidate trios consumed (TRIO stream index)
    uint32_t policy_ctr;   // random-policy steps taken (POLICY stream index)
};

#define BB_USED(s) (((s).pieces >> 24) & 7u)
#define BB_OVER(s) (((s).aux >> 16) & 1u)

struct BBRewardCfg {   // block_blast_env.py:63-71, order = oracle REWARD_KEYS
    double line_clear_base, block_placed, game_over_penalty, hole_penalty, center_bonus,
        combo_multiplier_bonus, survival_bonus;
};

#define BB_FLAG_RESEED_ON_RESET 1u   // reference behaviour when a seed is given (engine.py:137-138)
#define BB_FLAG_NO_AUTO_RESET 2u     // single-env semantics: stay in GAME_OVER (block_blast_env.py)

// exact float64 arithmetic without FMA contraction
BB_HD double bb_dmul(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    volatile double r = a * b; return r;
#endif
}
BB_HD double bb_dadd(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    volatile double r = a + b; return r;
#endif
}

// block_blast_env.py:158-193 (same operation order; result cast to f32 as wrappers.py:105)
BB_HD float bb_reward(const BBRewardCfg& c, int n_blocks, int lines, bool game_over,
                      int holes, int prev_holes, int center, int prev_center) {
    double r = bb_dadd(0.0, bb_dmul((double)n_blocks, c.block_placed));
    r = bb_dadd(r, c.survival_bonus);
    if (lines > 0) {
        const int cmul = lines < 4 ? lines : 4;
        double lr = bb_dmul((double)lines, c.line_clear_base);
        lr = bb_dmul(lr, (double)cmul);
        r = bb_dadd(r, lr);
        if (cmul > 1) r = bb_dadd(r, bb_dmul((double)(cmul - 1), c.combo_multiplier_bonus));
    }
    if (game_over) r = bb_dadd(r, c.game_over_penalty);
    const int d = holes - prev_holes;
    if (d > 0) r = bb_dadd(r, bb_dmul((double)d, c.hole_penalty));
    // openness = 1 - filled/16 is exact, so `openness >= prev` is `filled <= prev_filled`
    if (center <= prev_center) r = bb_dadd(r, bb_dmul(c.center_bonus, 0.1));
    return (float)r;
}

// draw until a solvable trio appears, at most 100 candidates (engine.py:155-172) — the
// sequential form; the step kernel runs the same loop warp-cooperatively (bb_warp_deal).
// Src: BBTrioSrc (the env's own stream / injected table) or BBLookaheadSrc (bb_env_expand).
template <class Src>
BB_HD uint32_t bb_deal(uint64_t board, const BBTables* T, const Src& src, uint64_t env_id, uint32_t* draw_ctr) {
    uint32_t trio = 0;
    for (int attempt = 0; attempt < 100; ++attempt) {
        trio = bb_candidate(src, env_id, *draw_ctr);
        *draw_ctr += 1;
        if (bb_solvable(board, T, trio)) break;
    }
    return trio;   // byte 3 = 0: nothing used
}

BB_HD void bb_reset_state(BBState& s, const BBTrioSrc& src, uint64_t env_id, uint32_t flags) {
    if (flags & BB_FLAG_RESEED_ON_RESET) s.draw_ctr = 0;
    s.board = 0;
    s.score = s.streak = s.moves = s.lines_total = s.max_streak = s.blocks_total = 0;
    s.aux = 0;             // prev_holes = 0, prev center filled = 0 (openness 1.0), not over
    // on an empty board every trio is solvable (checked exhaustively in tests), so the
    // first candidate is always accepted: engine.py:155-172 consumes exactly one draw
    s.pieces = bb_candidate(src, env_id, s.draw_ctr);
    s.draw_ctr += 1;
}

// the three action-mask planes of the current state (engine.py:364-380)
BB_HD void bb_action_mask(const BBState& s, const BBTables* T, uint64_t m[3]) {
    const uint64_t e = ~s.board;
    const uint32_t used = BB_USED(s);
    const bool over = BB_OVER(s);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const uint64_t v = bb_valid(e, bb_piece(T, (s.pieces >> (8 * i)) & 0xFFu));
        m[i] = (((used >> i) & 1u) || over) ? 0ull : v;
    }
}

struct BBStepOut {
    float reward;
    uint32_t terminated;   // 0/1
    uint32_t info;         // bit0 invalid, bits1-3 lines, 4-7 blocks, 8-10 combo mult, 11-17 draws, 18-31 score gained
    int32_t gain;          // score gained by this move
    int32_t ep_score, ep_len;   // valid when terminated
    uint64_t mask[3];      // action mask of the state after the step (after auto-reset)
};

struct BBMove { int n, lines, gain; bool ok, needs_deal; };

// Written only when an env terminates: what the reference keeps in infos[i] for a finished
// episode (block_blast_env.py:266-288 + terminal_observation, wrappers.py:97-100).  32 bytes.
struct BBEpisodeEnd {
    uint64_t board;            // terminal board
    uint32_t pieces;           // terminal trio + used bits
    int32_t lines_total, max_streak, blocks_total;
    uint32_t holes_fill;       // holes | filled cells << 8
    uint32_t last_move;        // the info word of the terminal move
};

// First half of a step: decode + validate (block_blast_env.py:104-118, :240-245,
// engine.py:326-346), place, clear, streak and score (engine.py:405-429).  On an invalid
// action the state is untouched and `o` is final (reward -10, mask of the unchanged state).
BB_HD BBMove bb_env_pre(BBState& s, int action, const BBTables* T, BBStepOut& o) {
    BBMove mv;
    mv.n = 0; mv.lines = 0; mv.gain = 0; mv.needs_deal = false;
    const uint32_t used = BB_USED(s);
    const int p = action >> 6;                 // action // 64 (negative actions -> p < 0)
    const int a = action & 63;
    bool ok = (action >= 0) && (p < 3) && !((used >> (p & 3)) & 1u) && !BB_OVER(s);
    const uint32_t id = ok ? ((s.pieces >> (8 * p)) & 0xFFu) : 0u;
    const uint64_t pm = T->row[id].mask;
    if (ok) ok = ((T->row[id].inb >> a) & 1ull) && (((pm << a) & s.board) == 0ull);
    mv.ok = ok;
    o.ep_score = 0; o.ep_len = 0; o.gain = 0;
    if (!ok) {
        o.reward = -10.0f;
        o.terminated = 0;
        o.info = 1u;
        bb_action_mask(s, T, o.mask);
        return mv;
    }
    const int n = (int)BB_META_N(T->row[id].meta);
    int lines;
    s.board = bb_clear(s.board | (pm << a), &lines);
    const uint32_t used2 = used | (1u << p);
    s.moves += 1;
    s.blocks_total += n;
    int gain = n;
    if (lines > 0) {
        s.streak += 1;
        s.max_streak = s.max_streak > s.streak ? s.max_streak : s.streak;
        s.lines_total += lines;
        const int cmul = lines < 4 ? lines : 4;
        const int smul = s.streak + 1 < 8 ? s.streak + 1 : 8;     // post-increment streak, engine.py:261
        gain += lines * 80 * cmul * smul;                         // lines*8 "blocks" x 10, engine.py:427
    } else {
        s.streak = 0;
    }
    s.score += gain;
    s.pieces = (s.pieces & 0x00FFFFFFu) | (used2 << 24);
    mv.n = n; mv.lines = lines; mv.gain = gain;
    mv.needs_deal = used2 == 7u;              // all three placed: regenerate (engine.py:432-437)
    return mv;
}

// Second half (after the deal, if any): game over iff no unused piece has an anchor
// (engine.py:440-441) — the same three valid masks are the next observation's action mask —
// then the shaped reward, and the vec-env's auto-reset (wrappers.py:96-102).
BB_HD void bb_env_post(BBState& s, const BBMove& mv, uint32_t draws, const BBTables* T, const BBRewardCfg& cfg,
                       const BBTrioSrc& src, uint64_t env_id, uint32_t flags, BBStepOut& o, BBEpisodeEnd* ep_end = nullptr) {
    bb_action_mask(s, T, o.mask);
    const bool over = (o.mask[0] | o.mask[1] | o.mask[2]) == 0ull;
    const int h = bb_holes(s.board), ctr = bb_center(s.board);
    o.reward = bb_reward(cfg, mv.n, mv.lines, over, h, (int)(s.aux & 0xFFu), ctr, (int)((s.aux >> 8) & 0xFFu));
    s.aux = (uint32_t)h | ((uint32_t)ctr << 8) | ((over ? 1u : 0u) << 16);
    o.terminated = over ? 1u : 0u;
    o.gain = mv.gain;
    // score gained <= 9 + 6*80*4*8 = 15,369 fits the 14 spare bits
    o.info = ((uint32_t)mv.lines << 1) | ((uint32_t)mv.n << 4) |
             ((uint32_t)(mv.lines > 0 ? (mv.lines < 4 ? mv.lines : 4) : 1) << 8) | (draws << 11) |
             ((uint32_t)mv.gain << 18);
    if (over) {
        o.ep_score = s.score;
        o.ep_len = s.moves;
        if (ep_end) {
            ep_end->board = s.board; ep_end->pieces = s.pieces;
            ep_end->lines_total = s.lines_total; ep_end->max_streak = s.max_streak; ep_end->blocks_total = s.blocks_total;
            ep_end->holes_fill = (uint32_t)h | ((uint32_t)bb_popc(s.board) << 8);
            ep_end->last_move = o.info;
        }
        if (!(flags & BB_FLAG_NO_AUTO_RESET)) {
            bb_reset_state(s, src, env_id, flags);
            // empty board, nothing used: every in-bounds anchor is valid
            o.mask[0] = T->row[s.pieces & 0xFFu].inb;
            o.mask[1] = T->row[(s.pieces >> 8) & 0xFFu].inb;
            o.mask[2] = T->row[(s.pieces >> 16) & 0xFFu].inb;
        }
    }
}

// One env step, sequential form (host build; the kernel composes pre / warp deal / post).
BB_HD void bb_env_apply(BBState& s, int action, const BBTables* T, const BBRewardCfg& cfg,
                        const BBTrioSrc& src, uint64_t env_id, uint32_t flags, BBStepOut& o) {
    const BBMove mv = bb_env_pre(s, action, T, o);
    if (!mv.ok) return;
    uint32_t draws = 0;
    if (mv.needs_deal) {
        const uint32_t before = s.draw_ctr;
        s.pieces = bb_deal(s.board, T, src, env_id, &s.draw_ctr);
        draws = s.draw_ctr - before;
    }
    bb_env_post(s, mv, draws, T, cfg, src, env_id, flags, o);
}

// k-th valid action (piece-major, then bit order = np.where(mask)[0] order,
// block_blast_env.py:313-323); k < number of valid actions
BB_HD int bb_kth_action(const uint64_t m[3], int k) {
    const int n0 = bb_popc(m[0]), n1 = bb_popc(m[1]);
    int p = 0;
    uint64_t w = m[0];
    if (k >= n0) { k -= n0; p = 1; w = m[1]; if (k >= n1) { k -= n1; p = 2; w = m[2]; } }
    return p * 64 + bb_select(w, k);
}

// the fused random-valid policy: k = mulhi(word, n_valid); 0 when nothing is valid
BB_HD int bb_pick_action(const uint64_t m[3], uint32_t word) {
    const int total = bb_popc(m[0]) + bb_popc(m[1]) + bb_popc(m[2]);
    if (total == 0) return 0;
    return bb_kth_action(m, (int)bb_mulhi(word, (uint32_t)total));
}

// ---------------------------------------------------------------------------------------
// bb_env_expand: the one-ply successors of a state.  Items of an env, in order: its valid actions
// in np.where(mask) order; when exactly one piece is left unused, every valid action places it and
// deals, and gives `samples` items (k = 0..samples-1) instead of one.  m = bb_action_mask(s), so a
// game-over state has no items.
// ---------------------------------------------------------------------------------------
BB_HD bool bb_expand_deals(const BBState& s) { return bb_popc32(BB_USED(s)) == 2; }

BB_HD int bb_expand_count(const BBState& s, const uint64_t m[3], int samples) {
    const int n = bb_popc(m[0]) + bb_popc(m[1]) + bb_popc(m[2]);
    return bb_expand_deals(s) ? n * samples : n;
}

// item j (0 <= j < bb_expand_count) -> action; *k = its sample index (0 for a non-deal item)
BB_HD int bb_expand_item(const BBState& s, const uint64_t m[3], int samples, int j, int* k) {
    int a = j;
    *k = 0;
    if (bb_expand_deals(s)) { a = j / samples; *k = j - a * samples; }
    return bb_kth_action(m, a);
}

// ---------------------------------------------------------------------------------------
// The 8 symmetries of the square (group D4).  The rules are invariant under all of them: the piece
// set is closed under each (BB_SYM_PERM), and placement, clears, score, holes, center openness and
// trio solvability only see cell sets.  Ids, as maps of cell (r, c):
//   0 identity (r, c)      1 R90 (c, 7-r)          2 R180 (7-r, 7-c)      3 R270 (7-c, r)
//   4 mirror columns (r, 7-c)   5 mirror rows (7-r, c)   6 transpose (c, r)   7 anti-transpose (7-c, 7-r)
// Each is "transpose, then mirror columns, then mirror rows", each step present or not: bit g of the
// masks below says whether symmetry g has that step.
// Pieces: the 8-bit ids of a pieces word map through BB_SYM_PERM (an id >= 37 stays as it is); slot
// order and used bits are kept.  Actions: slot*64 + a -> slot*64 + sigma_{g,p}(a), with
// sigma_{g,p}(a) = T_g(a) - BB_SYM_SHIFT[g][p]: the image of the top-left of the piece's bounding box
// minus the offset of the image box's top-left from it.  A legal anchor maps to a legal anchor of the
// image piece, so a mask plane maps as T_g(plane) >> shift (no wrap: every image anchor lies below
// and right of the shift).  Tables: tools/gen_piece_tables.py --sym.
// ---------------------------------------------------------------------------------------
#define BB_SYM_N 8
#define BB_SYM_HAS_TRANSPOSE 0xCAu     // g = 1, 3, 6, 7
#define BB_SYM_HAS_MIRROR_COLS 0x96u   // g = 1, 2, 4, 7
#define BB_SYM_HAS_MIRROR_ROWS 0xACu   // g = 2, 3, 5, 7

struct BBSymTables { uint8_t perm[BB_SYM_N][BB_TABLE_N]; uint8_t shift[BB_SYM_N][BB_TABLE_N]; };

static const uint8_t BB_HOST_SYM_PERM[BB_SYM_N][BB_TABLE_N] = BB_SYM_PERM;
static const uint8_t BB_HOST_SYM_SHIFT[BB_SYM_N][BB_TABLE_N] = BB_SYM_SHIFT;

inline void bb_fill_sym_tables(BBSymTables* t) {
    for (int g = 0; g < BB_SYM_N; ++g)
        for (int i = 0; i < BB_TABLE_N; ++i) { t->perm[g][i] = BB_HOST_SYM_PERM[g][i]; t->shift[g][i] = BB_HOST_SYM_SHIFT[g][i]; }
}

// (r, c) -> (c, r): three delta swaps
BB_HD uint64_t bb_transpose(uint64_t x) {
    uint64_t t = 0x0F0F0F0F00000000ull & (x ^ (x << 28)); x ^= t ^ (t >> 28);
    t = 0x3333000033330000ull & (x ^ (x << 14)); x ^= t ^ (t >> 14);
    t = 0x5500550055005500ull & (x ^ (x << 7)); x ^= t ^ (t >> 7);
    return x;
}
// (r, c) -> (7-r, c): byte swap
BB_HD uint64_t bb_mirror_rows(uint64_t x) {
#if defined(__CUDA_ARCH__)
    return (uint64_t)__byte_perm((uint32_t)(x >> 32), 0u, 0x0123u) | ((uint64_t)__byte_perm((uint32_t)x, 0u, 0x0123u) << 32);
#else
    return __builtin_bswap64(x);
#endif
}
// (r, c) -> (r, 7-c): bit reversal within each byte
BB_HD uint64_t bb_mirror_cols(uint64_t x) {
#if defined(__CUDA_ARCH__)
    // a 32-bit reversal takes (r, c) to (3-r, 7-c) within a half; a byte swap puts the rows back
    return (uint64_t)__byte_perm(__brev((uint32_t)x), 0u, 0x0123u) |
           ((uint64_t)__byte_perm(__brev((uint32_t)(x >> 32)), 0u, 0x0123u) << 32);
#else
    x = ((x >> 1) & 0x5555555555555555ull) | ((x & 0x5555555555555555ull) << 1);
    x = ((x >> 2) & 0x3333333333333333ull) | ((x & 0x3333333333333333ull) << 2);
    return ((x >> 4) & 0x0F0F0F0F0F0F0F0Full) | ((x & 0x0F0F0F0F0F0F0F0Full) << 4);
#endif
}

// T_g(board), 0 <= g < 8
BB_HD uint64_t bb_sym_board(int g, uint64_t b) {
    if ((BB_SYM_HAS_TRANSPOSE >> g) & 1u) b = bb_transpose(b);
    if ((BB_SYM_HAS_MIRROR_COLS >> g) & 1u) b = bb_mirror_cols(b);
    if ((BB_SYM_HAS_MIRROR_ROWS >> g) & 1u) b = bb_mirror_rows(b);
    return b;
}
// T_g of one cell index a = r*8 + c
BB_HD int bb_sym_cell(int g, int a) {
    int r = a >> 3, c = a & 7;
    if ((BB_SYM_HAS_TRANSPOSE >> g) & 1u) { const int t = r; r = c; c = t; }
    if ((BB_SYM_HAS_MIRROR_COLS >> g) & 1u) c = 7 - c;
    if ((BB_SYM_HAS_MIRROR_ROWS >> g) & 1u) r = 7 - r;
    return r * 8 + c;
}
// the pieces word of the transformed state: ids mapped, slot order and used bits kept
BB_HD uint32_t bb_sym_pieces(const BBSymTables* S, int g, uint32_t pw) {
    uint32_t out = pw & 0xFF000000u;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const uint32_t id = (pw >> (8 * k)) & 0xFFu;
        out |= (uint32_t)(id < BB_NUM_PIECES ? S->perm[g][id] : id) << (8 * k);
    }
    return out;
}
// sigma_{g,p}(a) for an in-bounds anchor a of piece `id` (< 37)
BB_HD int bb_sym_anchor(const BBSymTables* S, int g, uint32_t id, int a) {
    return bb_sym_cell(g, a) - (int)S->shift[g][id];
}
// the mask plane of a slot holding piece `id` (< 37) in the transformed state
BB_HD uint64_t bb_sym_mask_plane(const BBSymTables* S, int g, uint32_t id, uint64_t plane) {
    return bb_sym_board(g, plane) >> S->shift[g][id];
}
// the inverse of symmetry g (the two quarter turns swap, every other element is an involution)
BB_HD int bb_sym_inverse(int g) { return g == 1 ? 3 : g == 3 ? 1 : g; }
// Canonical representative of the orbit of (board b, pieces word pw): the view g with the smallest key
// (bb_sym_board(g, b) as u64, then bb_sym_pieces(g, pw) as u32; the full word, used bits and ids of used
// slots included).  Writes the view to *cb / *cp and returns the view set: bit g set iff view g equals it
// (never 0; its size is the order of the state's stabiliser).
BB_HD uint32_t bb_sym_canonical(const BBSymTables* S, uint64_t b, uint32_t pw, uint64_t* cb, uint32_t* cp) {
    uint64_t kb = b;
    uint32_t kp = pw, views = 1u;
#pragma unroll
    for (int g = 1; g < BB_SYM_N; ++g) {
        const uint64_t tb = bb_sym_board(g, b);
        const uint32_t tp = bb_sym_pieces(S, g, pw);
        if (tb < kb || (tb == kb && tp < kp)) { kb = tb; kp = tp; views = 1u << g; }
        else if (tb == kb && tp == kp) views |= 1u << g;
    }
    *cb = kb;
    *cp = kp;
    return views;
}
