// bb_env_kernels.cu — K1: the fused Block Blast env-step kernels for sm_100a.
//
// One thread owns one env.  The env state is 48 B kept as three 16-byte words in three SoA
// arrays (s0/s1/s2), so a warp reads and writes 3 x 512 contiguous bytes with 128-bit
// accesses; all outputs are SoA too (mask planes are plane-major).  The piece tables (40 x
// 32 B) are read from global memory through L1 (see g_bb_tables).
//
// Algorithmic HBM bytes per env-step (packed protocol, SURVEY.md §8d): state 48 R + 48 W,
// action 4, reward 4, terminated 1, mask 24  = 129 B.
//
// Reference path replaced: VectorizedBlockBlastEnv.step (src/environment/wrappers.py:75-116)
// -> BlockBlastEnv.step (src/environment/block_blast_env.py:224-264) -> GameEngine.make_move
// (src/game/engine.py:390-454); rules in bb_rules.cuh.
#include <cuda_runtime.h>
#include "bb_rules.cuh"
#include "bb_kernels.h"

// 40 rows of 32 bytes (the last three are zero padding), statically initialised in global memory.
// Lanes index the table with different piece ids, which constant memory would serialise; the 1.3 KB
// stay resident in L1, and reading them from there beat a per-block copy into shared memory
// (58.6 -> 57.2 us per launch: no staging loop, no barrier at block start).
__device__ BBTables g_bb_tables = {BB_PIECE_ROWS};

__device__ __forceinline__ void bb_load_state(const BBEnvArrays& E, int64_t i, BBState& s) {
    const uint4 a = E.s0[i], b = E.s1[i], c = E.s2[i];
    s.board = (uint64_t)a.x | ((uint64_t)a.y << 32);
    s.pieces = a.z;
    s.aux = a.w;
    s.score = (int32_t)b.x; s.streak = (int32_t)b.y; s.moves = (int32_t)b.z; s.lines_total = (int32_t)b.w;
    s.max_streak = (int32_t)c.x; s.blocks_total = (int32_t)c.y; s.draw_ctr = c.z; s.policy_ctr = c.w;
}

__device__ __forceinline__ void bb_store_state(const BBEnvArrays& E, int64_t i, const BBState& s) {
    E.s0[i] = make_uint4((uint32_t)s.board, (uint32_t)(s.board >> 32), s.pieces, s.aux);
    E.s1[i] = make_uint4((uint32_t)s.score, (uint32_t)s.streak, (uint32_t)s.moves, (uint32_t)s.lines_total);
    E.s2[i] = make_uint4((uint32_t)s.max_streak, (uint32_t)s.blocks_total, s.draw_ctr, s.policy_ctr);
}

__device__ __forceinline__ uint64_t bb_shfl64(uint64_t v, int src) {
    const uint32_t lo = __shfl_sync(0xffffffffu, (uint32_t)v, src);
    const uint32_t hi = __shfl_sync(0xffffffffu, (uint32_t)(v >> 32), src);
    return (uint64_t)lo | ((uint64_t)hi << 32);
}

// ---------------------------------------------------------------------------------------
// Warp-cooperative trio regeneration (engine.py:155-238).
//
// An env that placed its third piece must draw candidate trios until one is solvable (at
// most 100 draws, the last one is kept).  Candidate number d of env e is a pure function
// Philox(seed, e, d), so the warp evaluates candidates SPECULATIVELY IN PARALLEL instead of
// one after the other:
//   1. ballot the pending envs; split the 32 lanes into equal groups, one per pending env;
//      lane r of a group classifies candidate ctr + r of its env (bb_classify);
//   2. candidates that need a search (HARD) and come before the group's first provable
//      ACCEPT are resolved by the whole warp: lanes are re-split into teams, one per hard
//      item, each lane evaluates one branch of the search one unit at a time, and a ballot
//      after every unit stops a team as soon as one lane has proved solvability; teams are
//      re-formed until every item is decided (a lone heavy item ends up with all 32 lanes);
//   3. every group takes its first solvable candidate IN DRAW ORDER (or consumes all of its
//      candidates and goes round again), so the accepted trio and the advanced draw counter
//      are exactly those of the sequential loop.
// All 32 lanes of the warp must call this (lanes without work pass pending = false).
// ---------------------------------------------------------------------------------------
// Phase timers for tools/profile_phases.py (-DBB_PROFILE); BB_PF(...) vanishes in normal builds.
#ifdef BB_PROFILE
struct BBProf { long long cls = 0, team = 0, rounds = 0, iters = 0, t0 = 0, c0 = 0, c1 = 0, q0 = 0, q1 = 0, units = 0, units_all = 0, unit_cyc = 0; };
__device__ unsigned long long g_pf_units = 0, g_pf_units_max = 0, g_pf_open_cyc = 0, g_pf_unit_cyc = 0, g_pf_H = 0;
#define BB_PF(...) __VA_ARGS__
#else
struct BBProf {};
#define BB_PF(...)
#endif

// resolve the hard items of this warp; returns, for a lane that passed hard = true, whether
// its item (board it.b, pieces of `trio`) is solvable.
// Lane allocation is greedy over the concatenation of all items' remaining branches: an
// inclusive prefix sum of the remaining counts over the owner lanes maps worker lane L to
// (owner, branch) by binary search, so every round serves up to 32 branches whichever items they
// belong to (about ceil(sum of remaining branches / 32) rounds).  Measured against an equal split
// (32/#items lanes each, 90 us per launch) and a water-filling split (fewer rounds, 85 us): the
// greedy split is fastest (83 us) because fewer distinct items share a round, so the lanes of a
// warp run more coherent code.
__device__ __forceinline__ bool bb_warp_solve(bool hard, const BBItem& item, uint32_t trio, const BBTables* T,
                                              BBProf& pf) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    bool solved = false;
    uint32_t next = 0;                      // owner: first branch not yet handed out
    const uint32_t nbr = BB_PLAN_NA(item.plan) + BB_PLAN_NB(item.plan);
    unsigned hmask = __ballot_sync(FULL, hard);
    while (hmask) {
        BB_PF(pf.rounds += 1;)
        // Walk the hard lanes in order (a handful per round): their remaining branch counts laid
        // end to end are the round's work list, worker lane L serves entry L.  The shuffles of
        // this loop are independent of each other, unlike a prefix scan + binary search.
        const int rem = hard ? (int)(nbr - next) : 0;
        int excl = 32;                       // owner side: where MY item's branches start (32 = not served)
        int owner = lane, o_excl = 0, o_rem = 0;
        bool in_team = false;
        int run = 0;
        for (unsigned m = hmask; m && run < 32; m &= m - 1u) {
            const int h = __ffs((int)m) - 1;
            const int r = __shfl_sync(FULL, rem, h);
            if (lane == h) excl = run;
            if (lane >= run && lane < run + r) { owner = h; o_excl = run; o_rem = r; in_team = true; }
            run += r;
        }
        const int served_o = min(o_rem, 32 - o_excl);               // lanes working on my owner's item this round
        const unsigned team_mask = in_team ? ((served_o >= 32 ? FULL : ((1u << served_o) - 1u)) << o_excl) : 0u;
        BBItem it;
        it.b = bb_shfl64(item.b, owner);
        it.v[0] = bb_shfl64(item.v[0], owner);
        it.v[1] = bb_shfl64(item.v[1], owner);
        it.v[2] = bb_shfl64(item.v[2], owner);
        it.plan = __shfl_sync(FULL, item.plan, owner);
        const uint32_t tr = __shfl_sync(FULL, trio, owner);
        const uint32_t t = __shfl_sync(FULL, next, owner) + (uint32_t)(lane - o_excl);
        BBBranch br;
        br.bb = 0; br.m0 = 0; br.m1 = 0; br.always = 0;
        br.A.pm = br.A.inb = br.A.offs = 0; br.A.meta = 0;
        br.B = br.A;
        BB_PF(pf.q0 = clock64();)
        if (in_team) bb_branch_open(br, it, T, tr, t);              // t < nbr of the owner by construction
        BB_PF(pf.q1 = clock64(); pf.units = 0;)
        // unit loop: every lane advances its branch by one second-level anchor, then a
        // ballot tells each team whether one of its lanes has proved the trio solvable
        unsigned found = 0;                 // bit l set: lane l found a solution
        for (;;) {
            const bool work = in_team && !(found & team_mask) && ((br.m0 | br.m1) != 0ull);
            if (!__any_sync(FULL, work)) break;
            bool f = false;
            if (work) f = bb_branch_unit(br);
            found |= __ballot_sync(FULL, f);
            BB_PF(pf.units += 1;)
        }
        BB_PF(if (lane == 0) {
            pf.units_all += pf.units; pf.unit_cyc += clock64() - pf.q1;
            atomicAdd(&g_pf_units, (unsigned long long)pf.units);
            atomicMax(&g_pf_units_max, (unsigned long long)pf.units);
            atomicAdd(&g_pf_open_cyc, (unsigned long long)(pf.q1 - pf.q0));
            atomicAdd(&g_pf_unit_cyc, (unsigned long long)(clock64() - pf.q1));
            atomicAdd(&g_pf_H, (unsigned long long)__popc(hmask));
        })
        if (hard) {
            const int served = max(0, min(rem, 32 - excl));         // branches of MY item served this round
            const unsigned tm = served > 0 ? ((served >= 32 ? FULL : ((1u << served) - 1u)) << excl) : 0u;
            next += (uint32_t)served;
            if (found & tm) { hard = false; solved = true; }
            else if (next >= nbr) hard = false;                     // exhausted: not solvable
        }
        hmask = __ballot_sync(FULL, hard);
    }
    return solved;
}

// Src: where candidates come from (bb_candidate overloads in bb_rules.cuh) — BBTrioSrc for K1 (the env's
// own Philox stream or the injected table), BBLookaheadSrc for bb_env_expand.
template <class Src>
__device__ __forceinline__ uint32_t bb_warp_deal(bool pending, uint64_t board, const BBTables* T,
                                                 const Src& src, uint64_t env_id, uint32_t& pieces,
                                                 uint32_t& draw_ctr, BBProf& pf) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    uint32_t attempts = 0;                  // candidates consumed by MY env so far
    unsigned pmask = __ballot_sync(FULL, pending);
    while (pmask) {
        BB_PF(pf.c0 = clock64(); pf.iters += 1;)
        // 1. groups of w lanes, one group per pending env; lane r classifies candidate ctr + r
        const int P = __popc(pmask);
        const int w = 32 / P;
        const int g = lane / w, r = lane - g * w;
        const bool in_grp = g < P;
        const int owner = in_grp ? bb_select((uint64_t)pmask, g) : lane;
        const unsigned grp_bits = (w == 32 ? FULL : ((1u << w) - 1u));
        const int shift = (in_grp ? g : 0) * w;
        const uint64_t ob = bb_shfl64(board, owner);
        const uint64_t oid = bb_shfl64(env_id, owner);
        const uint32_t octr = __shfl_sync(FULL, draw_ctr, owner);
        const uint32_t oatt = __shfl_sync(FULL, attempts, owner);
        const bool cand = in_grp && (oatt + (uint32_t)r < 100u);
        BBItem item;
        item.b = ob; item.v[0] = item.v[1] = item.v[2] = 0; item.plan = 0;
        uint32_t trio = 0;
        int cls = BB_REJECT;
        if (cand) {
            trio = bb_candidate(src, oid, octr + (uint32_t)r);
            cls = bb_classify(ob, bb_piece(T, trio & 0xFFu), bb_piece(T, (trio >> 8) & 0xFFu),
                              bb_piece(T, (trio >> 16) & 0xFFu), &item);
        }
        // 2. hard candidates before the group's first provable accept need a search
        const unsigned amask = __ballot_sync(FULL, cls == BB_ACCEPT);
        const unsigned ga = (amask >> shift) & grp_bits;
        const int first_acc = ga ? (__ffs((int)ga) - 1) : w;
        const bool hard = cand && cls == BB_HARD && r < first_acc;
        BB_PF(pf.c1 = clock64(); pf.cls += pf.c1 - pf.c0;)
        const bool solved = bb_warp_solve(hard, item, trio, T, pf);
        BB_PF(pf.team += clock64() - pf.c1;)
        // 3. first solvable candidate of each group, in draw order
        const unsigned okmask = __ballot_sync(FULL, cand && (cls == BB_ACCEPT || solved));
        const unsigned go = (okmask >> shift) & grp_bits;
        const int nvalid = (int)min((uint32_t)w, 100u - oatt);          // candidates this group really had
        const int take = go ? __ffs((int)go) : nvalid;                  // draws consumed
        const bool done = go != 0u || (oatt + (uint32_t)take >= 100u);  // 100th failure: keep it (engine.py:171-172)
        const uint32_t chosen = __shfl_sync(FULL, trio, (in_grp ? g * w : 0) + take - 1);
        // hand the verdict to the env's own lane (which may sit in another group)
        const int my_base = pending ? __popc(pmask & ((1u << lane) - 1u)) * w : 0;
        const int t_take = __shfl_sync(FULL, take, my_base);
        const int t_done = __shfl_sync(FULL, (int)done, my_base);
        const uint32_t t_trio = __shfl_sync(FULL, chosen, my_base);
        if (pending) {
            draw_ctr += (uint32_t)t_take;
            attempts += (uint32_t)t_take;
            pieces = t_trio;                    // used bits cleared (engine.py:165)
            pending = !t_done;
        }
        pmask = __ballot_sync(FULL, pending);
    }
    return attempts;
}

// ---------------------------------------------------------------------------------------
// K1: one env step per thread; RANDOM fuses the uniform-random-valid policy and may run
// n_steps back to back with the state held in registers.
// ---------------------------------------------------------------------------------------
// INJECT: candidate trios come from the table of bb_env_set_trios (replay / parity runs) instead of
// Philox; a template parameter so that the production kernels do not carry the table pointer.
template <bool RANDOM, bool INJECT>
__global__ void __launch_bounds__(BB_STEP_THREADS, BB_STEP_MIN_BLOCKS)
bb_step_kernel(BBEnvArrays E, BBRewardCfg cfg, const int32_t* __restrict__ actions, int n_steps, int per_step,
               int32_t* __restrict__ actions_out, float* __restrict__ rewards,
               uint8_t* __restrict__ terminated, uint64_t* __restrict__ mask_out,
               int32_t* __restrict__ ep_score, int32_t* __restrict__ ep_len,
               uint32_t* __restrict__ info_out, unsigned long long* __restrict__ stats,
               uint64_t* __restrict__ board_out, uint32_t* __restrict__ pieces_out,
               const uint64_t* __restrict__ mask_in) {
    const BBTables& T = g_bb_tables;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < E.n;
    unsigned st_eps = 0, st_score = 0, st_len = 0, st_max = 0;   // per thread, 32 bits: n_steps <= 2^20 (API check)
    BBTrioSrc src(E.seed);
    if (INJECT) { src.trios = E.trios; src.len = E.trio_len; src.base = E.trio_base; }
    BBState s;
    BBStepOut o;
    int action = 0;
    const uint64_t env_id = (uint64_t)(E.env_offset + (live ? i : 0));
    if (live) {
        bb_load_state(E, i, s);
        if (RANDOM) {
            if (mask_in) {
                // the caller hands back the mask the previous step / reset wrote for this state
                const int64_t ms = E.out_stride ? E.out_stride : E.n;
                o.mask[0] = mask_in[i]; o.mask[1] = mask_in[ms + i]; o.mask[2] = mask_in[2 * ms + i];
            } else {
                bb_action_mask(s, &T, o.mask);
            }
        } else {
            action = actions[i];
        }
    } else {
        s.board = 0; s.pieces = 0; s.aux = 0; s.draw_ctr = 0; s.policy_ctr = 0;
        s.score = s.streak = s.moves = s.lines_total = s.max_streak = s.blocks_total = 0;
        o.mask[0] = o.mask[1] = o.mask[2] = 0;
    }
    const int steps = RANDOM ? n_steps : 1;
    BBProf pf;
    BB_PF(pf.t0 = clock64();)
    for (int step = 0; step < steps; ++step) {
        BBMove mv;
        mv.ok = false; mv.needs_deal = false; mv.n = 0; mv.lines = 0; mv.gain = 0;
        if (live) {
            if (RANDOM) {
                const BBPhilox4 r = bb_philox((uint32_t)env_id, (uint32_t)(env_id >> 32), s.policy_ctr,
                                              BB_STREAM_POLICY, (uint32_t)E.seed, (uint32_t)(E.seed >> 32));
                s.policy_ctr += 1;
                action = bb_pick_action(o.mask, r.x);
            }
            mv = bb_env_pre(s, action, &T, o);
        }
        // all 32 lanes take part in the deal, with or without work of their own
        const uint32_t draws = bb_warp_deal(live && mv.ok && mv.needs_deal, s.board, &T, src, env_id,
                                            s.pieces, s.draw_ctr, pf);
        if (live && mv.ok) {
            bb_env_post(s, mv, draws, &T, cfg, src, env_id, E.flags, o, E.ep_end ? E.ep_end + i : nullptr);
            if (o.terminated) {
                st_eps += 1u; st_score += (unsigned)o.ep_score; st_len += (unsigned)o.ep_len;
                st_max = max(st_max, (unsigned)o.ep_score);
            }
        }
        if (RANDOM && per_step && live) {
            // rollout mode: every step's outputs go to row `step` of [n_steps][...] arrays
            const int64_t base = (int64_t)step * E.n + i;
            if (actions_out) actions_out[base] = action;
            if (rewards) rewards[base] = o.reward;
            if (terminated) terminated[base] = (uint8_t)o.terminated;
            if (mask_out) {
                const int64_t mb = (int64_t)step * 3 * E.n + i;
                mask_out[mb] = o.mask[0];
                mask_out[mb + E.n] = o.mask[1];
                mask_out[mb + 2 * E.n] = o.mask[2];
            }
        }
    }
    if (RANDOM && per_step) {
        if (live) bb_store_state(E, i, s);
        actions_out = nullptr; rewards = nullptr; terminated = nullptr; mask_out = nullptr;   // already written
    }
    if (live) {
        if (!(RANDOM && per_step)) bb_store_state(E, i, s);
        if (RANDOM && actions_out) actions_out[i] = action;
        if (rewards) rewards[i] = o.reward;
        if (terminated) terminated[i] = (uint8_t)o.terminated;
        if (mask_out) {
            const int64_t ms = E.out_stride ? E.out_stride : E.n;
            mask_out[i] = o.mask[0];
            mask_out[ms + i] = o.mask[1];
            mask_out[2 * ms + i] = o.mask[2];
        }
        if (o.terminated) {
            if (ep_score) ep_score[i] = o.ep_score;
            if (ep_len) ep_len[i] = o.ep_len;
        }
        if (info_out) info_out[i] = o.info;
        if (board_out) board_out[i] = s.board;          // the next observation (packed)
        if (pieces_out) pieces_out[i] = s.pieces;
    }
    if (stats) {
        // warp-reduce with redux.sync (16-bit limbs of the score sum so that 32 lanes cannot wrap),
        // one atomic per warp per counter
        const unsigned FULLM = 0xffffffffu;
        const unsigned long long w_eps = __reduce_add_sync(FULLM, st_eps);
        const unsigned long long w_score = (unsigned long long)__reduce_add_sync(FULLM, st_score & 0xFFFFu) +
                                           ((unsigned long long)__reduce_add_sync(FULLM, st_score >> 16) << 16);
        const unsigned long long w_len = (unsigned long long)__reduce_add_sync(FULLM, st_len & 0xFFFFu) +
                                         ((unsigned long long)__reduce_add_sync(FULLM, st_len >> 16) << 16);
        const unsigned w_max = __reduce_max_sync(FULLM, st_max);
        const unsigned long long nlive = __popc(__ballot_sync(0xffffffffu, live));
        if ((threadIdx.x & 31) == 0) {
            BB_PF(const unsigned long long tot = (unsigned long long)(clock64() - pf.t0);
                  atomicAdd(&stats[4], tot);
                  atomicAdd(&stats[5], (unsigned long long)pf.cls);
                  atomicAdd(&stats[6], (unsigned long long)pf.team);
                  atomicAdd(&stats[7], (unsigned long long)pf.rounds);
                  atomicAdd(&stats[8], (unsigned long long)pf.iters);
                  atomicMax(&stats[9], tot);
                  atomicMax(&stats[10], (unsigned long long)pf.rounds);
                  // heaviest warps: cycles << 32 | unit-loop cycles/64 << 16 | unit iterations << 8 | rounds
                  atomicMax(&stats[63 - (tot & 7)], (tot << 32) | (((unsigned long long)pf.unit_cyc >> 6) << 16) |
                                                        ((unsigned long long)(pf.units_all > 255 ? 255 : pf.units_all) << 8) | (unsigned long long)(pf.rounds > 255 ? 255 : pf.rounds));
                  stats[11] = g_pf_units; stats[12] = g_pf_units_max; stats[13] = g_pf_open_cyc;
                  stats[14] = g_pf_unit_cyc; stats[15] = g_pf_H;
                  atomicAdd(&stats[16 + (tot >> 13 > 31 ? 31 : tot >> 13)], 1ull);           // cycles histogram
                  atomicAdd(&stats[48 + (pf.rounds > 7 ? 7 : pf.rounds)], 1ull);)           // rounds histogram
            atomicAdd(&stats[0], nlive * (unsigned long long)n_steps);
            if (w_eps) {
                atomicAdd(&stats[1], w_eps);
                atomicAdd(&stats[2], w_score);
                atomicAdd(&stats[3], w_len);
#ifndef BB_PROFILE
                atomicMax(&stats[4], (unsigned long long)w_max);
#endif
            }
        }
    }
}

// ---------------------------------------------------------------------------------------
// reset (VectorizedBlockBlastEnv.reset, wrappers.py:53-73) and observe
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(BB_STEP_THREADS)
bb_reset_kernel(BBEnvArrays E, const uint8_t* __restrict__ reset_mask, uint64_t* __restrict__ mask_out) {
    const BBTables& T = g_bb_tables;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= E.n) return;
    BBState s;
    bb_load_state(E, i, s);
    if (!reset_mask || reset_mask[i]) {
        BBTrioSrc src(E.seed);
        src.trios = E.trios; src.len = E.trio_len; src.base = E.trio_base;
        bb_reset_state(s, src, (uint64_t)(E.env_offset + i), E.flags);
        bb_store_state(E, i, s);
    }
    if (mask_out) {
        uint64_t m[3];
        bb_action_mask(s, &T, m);
        mask_out[i] = m[0];
        mask_out[E.n + i] = m[1];
        mask_out[2 * E.n + i] = m[2];
    }
}

__global__ void __launch_bounds__(BB_STEP_THREADS)
bb_observe_kernel(BBEnvArrays E, uint64_t* __restrict__ board_out, uint32_t* __restrict__ pieces_out,
                  uint64_t* __restrict__ mask_out) {
    const BBTables& T = g_bb_tables;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= E.n) return;
    BBState s;
    bb_load_state(E, i, s);
    if (board_out) board_out[i] = s.board;
    if (pieces_out) pieces_out[i] = s.pieces;
    if (mask_out) {
        uint64_t m[3];
        bb_action_mask(s, &T, m);
        mask_out[i] = m[0];
        mask_out[E.n + i] = m[1];
        mask_out[2 * E.n + i] = m[2];
    }
}

// uniform random valid action of the current state (sample_valid_actions, wrappers.py:133-136):
// k-th set bit of the 192-bit mask, k = mulhi(word, n_valid); 0 when nothing is valid.  Uses
// Philox stream 3 with a caller-supplied call counter; the env state is not modified.
#define BB_STREAM_SAMPLE_VALID 3u
__global__ void __launch_bounds__(BB_STEP_THREADS)
bb_sample_valid_kernel(BBEnvArrays E, uint64_t call_counter, int32_t* __restrict__ actions_out) {
    const BBTables& T = g_bb_tables;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= E.n) return;
    BBState s;
    bb_load_state(E, i, s);
    uint64_t m[3];
    bb_action_mask(s, &T, m);
    const uint64_t env_id = (uint64_t)(E.env_offset + i);
    const BBPhilox4 r = bb_philox((uint32_t)env_id, (uint32_t)(env_id >> 32), (uint32_t)call_counter,
                                  BB_STREAM_SAMPLE_VALID, (uint32_t)E.seed, (uint32_t)(E.seed >> 32));
    actions_out[i] = bb_pick_action(m, r.x);
}

// ---------------------------------------------------------------------------------------
// bb_env_expand: one-ply successors of every env's current state (bb_expand_* in bb_rules.cuh).
// Phase 1 counts the items of each env and scans the counts into offsets[n+1] (three launches: a
// block-local scan, a one-block scan of the block totals, the add); phase 2 runs one lane per item.
// Nothing of the env state is written.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ int64_t bb_warp_incl_scan(int64_t v) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int64_t u = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += u;
    }
    return v;
}

// inclusive scan over the block (blockDim.x = BB_STEP_THREADS); *total = the block's sum
__device__ __forceinline__ int64_t bb_block_incl_scan(int64_t v, int64_t* total) {
    __shared__ int64_t warp_sums[BB_STEP_THREADS / 32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    v = bb_warp_incl_scan(v);
    if (lane == 31) warp_sums[w] = v;
    __syncthreads();
    if (w == 0) {
        int64_t t = lane < BB_STEP_THREADS / 32 ? warp_sums[lane] : 0;
        t = bb_warp_incl_scan(t);
        if (lane < BB_STEP_THREADS / 32) warp_sums[lane] = t;
    }
    __syncthreads();
    if (w > 0) v += warp_sums[w - 1];
    *total = warp_sums[BB_STEP_THREADS / 32 - 1];
    __syncthreads();
    return v;
}

// offsets[i] = exclusive scan of env i's item count within its block; block_sums[b] = block total
__global__ void __launch_bounds__(BB_STEP_THREADS)
bb_expand_count_kernel(BBEnvArrays E, int samples, int64_t* __restrict__ offsets, int64_t* __restrict__ block_sums) {
    const BBTables& T = g_bb_tables;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t c = 0;
    if (i < E.n) {
        BBState s;
        bb_load_state(E, i, s);
        uint64_t m[3];
        bb_action_mask(s, &T, m);
        c = bb_expand_count(s, m, samples);
    }
    int64_t total;
    const int64_t incl = bb_block_incl_scan(c, &total);
    if (i < E.n) offsets[i] = incl - c;
    if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

// one block: block_sums[0..nb) -> exclusive scan in place; offsets[n] = grand total
__global__ void __launch_bounds__(BB_STEP_THREADS)
bb_expand_scan_blocks_kernel(int64_t* __restrict__ block_sums, int64_t nb, int64_t* __restrict__ offsets_end) {
    int64_t carry = 0;
    for (int64_t base = 0; base < nb; base += BB_STEP_THREADS) {
        const int64_t j = base + threadIdx.x;
        const int64_t v = j < nb ? block_sums[j] : 0;
        int64_t total;
        const int64_t incl = bb_block_incl_scan(v, &total);
        if (j < nb) block_sums[j] = carry + incl - v;
        carry += total;
    }
    if (threadIdx.x == 0) *offsets_end = carry;
}

__global__ void __launch_bounds__(BB_STEP_THREADS)
bb_expand_add_kernel(int64_t n, const int64_t* __restrict__ block_sums, int64_t* __restrict__ offsets) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) offsets[i] += block_sums[blockIdx.x];
}

// Phase 2: lane = item.  Items of one env are adjacent, so the deals of a state with one piece left
// (all of its items) share warps — the many-pending case bb_warp_deal spreads over the lanes.
__global__ void __launch_bounds__(BB_STEP_THREADS, BB_STEP_MIN_BLOCKS)
bb_expand_kernel(BBEnvArrays E, BBRewardCfg cfg, uint32_t call_counter, int samples, int64_t capacity,
                 const int64_t* __restrict__ offsets, int32_t* __restrict__ action_out, float* __restrict__ reward_out,
                 uint8_t* __restrict__ terminated_out, uint32_t* __restrict__ info_out,
                 uint64_t* __restrict__ board_out, uint32_t* __restrict__ pieces_out, uint64_t* __restrict__ mask_out) {
    const BBTables& T = g_bb_tables;
    const int64_t item = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t n = E.n;
    const bool live = item < capacity && item < offsets[n];
    BBState s;
    s.board = 0; s.pieces = 0; s.aux = 0; s.draw_ctr = 0; s.policy_ctr = 0;
    s.score = s.streak = s.moves = s.lines_total = s.max_streak = s.blocks_total = 0;
    BBStepOut o;
    BBMove mv;
    mv.ok = false; mv.needs_deal = false; mv.n = 0; mv.lines = 0; mv.gain = 0;
    int action = 0, k = 0;
    uint64_t env_id = 0;
    if (live) {
        int64_t lo = 0, hi = n;                       // offsets[lo] <= item < offsets[hi]
        while (hi - lo > 1) {
            const int64_t mid = (lo + hi) >> 1;
            if (offsets[mid] <= item) lo = mid; else hi = mid;
        }
        env_id = (uint64_t)(E.env_offset + lo);
        bb_load_state(E, lo, s);
        uint64_t m[3];
        bb_action_mask(s, &T, m);
        action = bb_expand_item(s, m, samples, (int)(item - offsets[lo]), &k);
        mv = bb_env_pre(s, action, &T, o);
    }
    BBLookaheadSrc src;
    src.seed = E.seed; src.call_counter = call_counter;
    uint32_t draw = (uint32_t)k << 8;                 // LOOKAHEAD candidate index k << 8 | d (bb_rules.cuh)
    BBProf pf;
    const uint32_t draws = bb_warp_deal(live && mv.ok && mv.needs_deal, s.board, &T, src, env_id, s.pieces, draw, pf);
    if (!live) return;
    bb_env_post(s, mv, draws, &T, cfg, BBTrioSrc(E.seed), env_id, BB_FLAG_NO_AUTO_RESET, o);
    if (action_out) action_out[item] = action;
    if (reward_out) reward_out[item] = o.reward;
    if (terminated_out) terminated_out[item] = (uint8_t)o.terminated;
    if (info_out) info_out[item] = o.info;
    if (board_out) board_out[item] = s.board;
    if (pieces_out) pieces_out[item] = s.pieces;
    if (mask_out) {
        mask_out[item] = o.mask[0];
        mask_out[capacity + item] = o.mask[1];
        mask_out[2 * capacity + item] = o.mask[2];
    }
}

// ---------------------------------------------------------------------------------------
// bb_env_observe_live: the observation of every env that is not game over, compacted into rows
// 0..count-1 in ascending env order.  Count per block -> bb_expand_scan_blocks_kernel (exclusive
// block offsets, grand total) -> write; no atomics, so the row order is fixed.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(BB_STEP_THREADS)
bb_live_count_kernel(BBEnvArrays E, int64_t* __restrict__ block_sums) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < E.n && !((E.s0[i].w >> 16) & 1u);       // aux byte 2: game over (BB_OVER)
    const int c = __syncthreads_count(live);
    if (threadIdx.x == 0) block_sums[blockIdx.x] = c;
}

// row of env i = its block's offset + live envs before it in the block (warp ballots)
__global__ void __launch_bounds__(BB_STEP_THREADS)
bb_observe_live_kernel(BBEnvArrays E, const int64_t* __restrict__ block_offsets, const int64_t* __restrict__ total,
                       uint64_t* __restrict__ board_out, uint32_t* __restrict__ pieces_out, uint64_t* __restrict__ mask_out,
                       int64_t mask_stride, int32_t* __restrict__ ids_out, int32_t* __restrict__ count_out) {
    __shared__ int warp_live[BB_STEP_THREADS / 32];
    const BBTables& T = g_bb_tables;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    BBState s;
    bool live = false;
    if (i < E.n) {
        bb_load_state(E, i, s);
        live = !BB_OVER(s);
    }
    const unsigned ballot = __ballot_sync(0xffffffffu, live);
    if (lane == 0) warp_live[w] = __popc(ballot);
    __syncthreads();
    int before = __popc(ballot & ((1u << lane) - 1u));
    for (int k = 0; k < w; ++k) before += warp_live[k];
    if (i == 0) *count_out = (int32_t)*total;
    if (!live) return;
    const int64_t row = block_offsets[blockIdx.x] + before;
    board_out[row] = s.board;
    pieces_out[row] = s.pieces;
    uint64_t m[3];
    bb_action_mask(s, &T, m);
    mask_out[row] = m[0];
    mask_out[mask_stride + row] = m[1];
    mask_out[2 * mask_stride + row] = m[2];
    ids_out[row] = (int32_t)i;
}

// ---------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------
static inline unsigned bb_grid(int64_t n) { return (unsigned)((n + BB_STEP_THREADS - 1) / BB_STEP_THREADS); }

// one int64 per block of the offset scan, plus the grand total of bb_launch_observe_live's scan
int64_t bb_expand_scratch_count(int64_t n) { return (int64_t)bb_grid(n) + 1; }

cudaError_t bb_launch_observe_live(const BBEnvArrays& E, int64_t* scratch, uint64_t* board_out, uint32_t* pieces_out,
                                   uint64_t* mask_out, int64_t mask_stride, int32_t* ids_out, int32_t* count_out,
                                   cudaStream_t stream) {
    const unsigned nb = bb_grid(E.n);
    bb_live_count_kernel<<<nb, BB_STEP_THREADS, 0, stream>>>(E, scratch);
    bb_expand_scan_blocks_kernel<<<1, BB_STEP_THREADS, 0, stream>>>(scratch, (int64_t)nb, scratch + nb);
    bb_observe_live_kernel<<<nb, BB_STEP_THREADS, 0, stream>>>(E, scratch, scratch + nb, board_out, pieces_out, mask_out,
                                                               mask_stride, ids_out, count_out);
    return cudaGetLastError();
}

cudaError_t bb_launch_expand(const BBEnvArrays& E, const BBRewardCfg& cfg, uint32_t call_counter, int samples,
                             int64_t capacity, int64_t* offsets, int64_t* scratch, int32_t* action_out, float* reward_out,
                             uint8_t* terminated_out, uint32_t* info_out, uint64_t* board_out, uint32_t* pieces_out,
                             uint64_t* mask_out, cudaStream_t stream) {
    const unsigned nb = bb_grid(E.n);
    bb_expand_count_kernel<<<nb, BB_STEP_THREADS, 0, stream>>>(E, samples, offsets, scratch);
    bb_expand_scan_blocks_kernel<<<1, BB_STEP_THREADS, 0, stream>>>(scratch, (int64_t)nb, offsets + E.n);
    bb_expand_add_kernel<<<nb, BB_STEP_THREADS, 0, stream>>>(E.n, scratch, offsets);
    if (capacity > 0)
        bb_expand_kernel<<<bb_grid(capacity), BB_STEP_THREADS, 0, stream>>>(
            E, cfg, call_counter, samples, capacity, offsets, action_out, reward_out, terminated_out, info_out, board_out,
            pieces_out, mask_out);
    return cudaGetLastError();
}

cudaError_t bb_launch_step(const BBEnvArrays& E, const BBRewardCfg& cfg, const int32_t* actions,
                           float* rewards, uint8_t* terminated, uint64_t* mask_out, uint64_t* board_out,
                           uint32_t* pieces_out, int32_t* ep_score, int32_t* ep_len, uint32_t* info_out,
                           unsigned long long* stats, cudaStream_t stream) {
    if (E.trios)
        bb_step_kernel<false, true><<<bb_grid(E.n), BB_STEP_THREADS, 0, stream>>>(
            E, cfg, actions, 1, 0, nullptr, rewards, terminated, mask_out, ep_score, ep_len, info_out, stats, board_out,
            pieces_out, nullptr);
    else
        bb_step_kernel<false, false><<<bb_grid(E.n), BB_STEP_THREADS, 0, stream>>>(
            E, cfg, actions, 1, 0, nullptr, rewards, terminated, mask_out, ep_score, ep_len, info_out, stats, board_out,
            pieces_out, nullptr);
    return cudaGetLastError();
}

cudaError_t bb_launch_step_range(const BBEnvArrays& E, const BBRewardCfg& cfg, int64_t off, int64_t cnt,
                                 const int32_t* actions, float* rewards, uint8_t* terminated, uint64_t* mask_out,
                                 int32_t* ep_score, int32_t* ep_len, uint32_t* info_out, uint64_t* board_out,
                                 uint32_t* pieces_out, cudaStream_t stream) {
    if (cnt <= 0) return cudaSuccess;
    BBEnvArrays R = E;
    R.s0 += off; R.s1 += off; R.s2 += off;
    R.n = cnt;
    R.env_offset += off;
    if (R.ep_end) R.ep_end += off;
    R.out_stride = E.n;
#define BB_OFF(p) ((p) ? (p) + off : nullptr)
    if (R.trios)
        bb_step_kernel<false, true><<<bb_grid(cnt), BB_STEP_THREADS, 0, stream>>>(
            R, cfg, actions + off, 1, 0, nullptr, BB_OFF(rewards), BB_OFF(terminated), BB_OFF(mask_out), BB_OFF(ep_score),
            BB_OFF(ep_len), BB_OFF(info_out), nullptr, BB_OFF(board_out), BB_OFF(pieces_out), nullptr);
    else
        bb_step_kernel<false, false><<<bb_grid(cnt), BB_STEP_THREADS, 0, stream>>>(
            R, cfg, actions + off, 1, 0, nullptr, BB_OFF(rewards), BB_OFF(terminated), BB_OFF(mask_out), BB_OFF(ep_score),
            BB_OFF(ep_len), BB_OFF(info_out), nullptr, BB_OFF(board_out), BB_OFF(pieces_out), nullptr);
#undef BB_OFF
    return cudaGetLastError();
}

cudaError_t bb_launch_step_random(const BBEnvArrays& E, const BBRewardCfg& cfg, int n_steps, int per_step,
                                  int32_t* actions_out, float* rewards, uint8_t* terminated,
                                  uint64_t* mask_out, unsigned long long* stats, const uint64_t* mask_in,
                                  cudaStream_t stream) {
    if (E.trios)
        bb_step_kernel<true, true><<<bb_grid(E.n), BB_STEP_THREADS, 0, stream>>>(
            E, cfg, nullptr, n_steps, per_step, actions_out, rewards, terminated, mask_out, nullptr, nullptr, nullptr, stats,
            nullptr, nullptr, mask_in);
    else
        bb_step_kernel<true, false><<<bb_grid(E.n), BB_STEP_THREADS, 0, stream>>>(
            E, cfg, nullptr, n_steps, per_step, actions_out, rewards, terminated, mask_out, nullptr, nullptr, nullptr, stats,
            nullptr, nullptr, mask_in);
    return cudaGetLastError();
}

// a new injected trio table restarts every env's candidate stream at draw 0
__global__ void bb_zero_draw_ctr_kernel(BBEnvArrays E) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < E.n) E.s2[i].z = 0u;
}

cudaError_t bb_launch_zero_draw_ctr(const BBEnvArrays& E, cudaStream_t stream) {
    bb_zero_draw_ctr_kernel<<<bb_grid(E.n), BB_STEP_THREADS, 0, stream>>>(E);
    return cudaGetLastError();
}

cudaError_t bb_launch_reset(const BBEnvArrays& E, const uint8_t* reset_mask, uint64_t* mask_out, cudaStream_t stream) {
    bb_reset_kernel<<<bb_grid(E.n), BB_STEP_THREADS, 0, stream>>>(E, reset_mask, mask_out);
    return cudaGetLastError();
}

cudaError_t bb_launch_observe(const BBEnvArrays& E, uint64_t* board_out, uint32_t* pieces_out,
                              uint64_t* mask_out, cudaStream_t stream) {
    bb_observe_kernel<<<bb_grid(E.n), BB_STEP_THREADS, 0, stream>>>(E, board_out, pieces_out, mask_out);
    return cudaGetLastError();
}

cudaError_t bb_launch_sample_valid(const BBEnvArrays& E, uint64_t call_counter, int32_t* actions_out, cudaStream_t stream) {
    bb_sample_valid_kernel<<<bb_grid(E.n), BB_STEP_THREADS, 0, stream>>>(E, call_counter, actions_out);
    return cudaGetLastError();
}
