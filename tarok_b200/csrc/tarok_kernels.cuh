// sm_100a kernels of the batched Tarok environment.
//
// HBM layout (structure of arrays, one 64-bit word per game per field, n_alloc = n rounded up to
// the 512-game CTA tile, every array 256-byte aligned):
//   hands[4][n_alloc] (leader-relative slots, see "hand slots" below; everything else is indexed by seat)
//   piles[4][n_alloc]  talon[n_alloc]  torder[n_alloc]  meta[n_alloc]
//   mask[n_alloc]  scores[n_alloc] (int16 x4)  tricklog[12][n_alloc] (uint32)  dpts[n_alloc] (uint8)
//   optional (TAROK_FLAG_HISTORY): hist[48][n_alloc] (uint8)  hands0[4][n_alloc]  discard[n_alloc]  qmax_hist[48][n_alloc] (float)
// The stepwise kernels give each lane TWO consecutive games so that every per-field access is one
// 128-bit load/store (ld.global.v2.u64): a warp covers a 64-game tile = 512 contiguous bytes per
// field.  Per-game logic is branch-light integer code (popc / shifts / selects, tarok_rules.cuh).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

#include "philox.cuh"
#include "tarok_rules.cuh"

namespace tk {

#ifndef TK_CTA
#define TK_CTA 256
#endif
constexpr int CTA = TK_CTA;
constexpr int TILE = 2 * CTA;          // games per CTA in the 2-games-per-lane kernels

// Resident CTAs per SM the register allocation is bounded for (A/B-measured on B200, profiles/r02/occupancy_ab.md; the
// macros exist so that a variant library can be built with other bounds: python -m tarok_b200.build --variant ...).
#ifndef TK_STEP_BLOCKS_RANDOM
#define TK_STEP_BLOCKS_RANDOM 5   // 48 registers, trick positions 0-2 and the general path: 69.2 -> 66.1 us at 8 M deals, = at 1 M
#endif
#ifndef TK_STEP_BLOCKS_RANDOM_012
#define TK_STEP_BLOCKS_RANDOM_012 TK_STEP_BLOCKS_RANDOM   // trick positions 0-2 (lighter than the trick-closing one)
#endif
#ifndef TK_STEP_BLOCKS_RANDOM_3
#define TK_STEP_BLOCKS_RANDOM_3 4 // the trick-closing position: 64 registers, no spills; at 5 blocks (48 registers) it spilled
#endif                            // 32 / 64 B: headline 0.4575 -> 0.4434 ms per rollout at 1 M deals (profiles/r03)
#ifndef TK_STEP_BLOCKS_FORCED
#define TK_STEP_BLOCKS_FORCED 5   // 46-48 registers: 8.63 -> 8.22 us per launch at 1 M deals (6 blocks = 40 registers spills and loses)
#endif
#ifndef TK_STEP_BLOCKS_BOTS
#define TK_STEP_BLOCKS_BOTS 4     // tarok_step_bots: the forced path plus a Philox block and a pick; 64 registers keep it spill-free
#endif
#ifndef TK_SETUP_BLOCKS
#define TK_SETUP_BLOCKS 3
#endif

struct Env {
    u64* hands; u64* piles; u64* talon; u64* torder; u64* meta; u64* mask; u64* scores;
    uint8_t* hist; u64* hands0; u64* discard; float* qmax_hist; long long* stats;
    u32* tricklog;                         // [12][n_alloc]: trick k of game g = 4 cards (24 bit, play order) | card points << 24 | called-king flag << 29 | winner << 30
    uint8_t* dpts;                         // [n_alloc]: card points of the declarer's discards (scoring reads this instead of the piles)
    uint2* rcache;                         // [3][n_alloc / 2] draw cache: {tag, the pair's 16-bit lanes of trick position 1 + row}
    u32 rc_epoch;                          // high bits of a valid tag: bumped whenever first_gid is (re)set; low 4 bits = trick
    u32 rc_rows;                           // trick positions 1..rc_rows use the cache (0 = off, 2, 3): TAROK_OPT_DRAW_CACHE
    u64 n, n_alloc, first_gid;
    Rng rng;                               // seed + precomputed Philox round keys
    const struct RunParams* run_ptr;       // device record the GRAPH kernel variants take first_gid / rc_epoch from
};

// What changes from one rollout to the next.  Kernel parameters are frozen into a captured CUDA graph, so the kernels of a
// graph-backed rollout (tarok_rollout_stepwise, TAROK_OPT_GRAPH; template parameter GRAPH) read these two from a 16-byte
// device record that a one-thread kernel (k_set_run) rewrites in stream order before every replay.
struct RunParams { u64 first_gid; u32 rc_epoch; u32 pad; };
// GRAPH kernels overwrite their own copy of the two fields first thing (kernel parameters are ordinary local variables), so
// every helper below keeps reading e.first_gid / e.rc_epoch and the plain kernels carry no trace of the indirection.
__device__ __forceinline__ void load_run_params(Env& e) {
    const uint4 rp = __ldg(reinterpret_cast<const uint4*>(e.run_ptr));
    e.first_gid = (u64)rp.x | ((u64)rp.y << 32);
    e.rc_epoch = rp.z;
}
__global__ void k_set_run(RunParams* r, u64 first_gid, u32 rc_epoch) { r->first_gid = first_gid; r->rc_epoch = rc_epoch; r->pad = 0u; }

enum : int { S_SEAT = 0, S_PLAYER = 4, S_CONTRACT = 8, S_FINISHED = 18, S_STEPS = 19, S_ERRORS = 20, S_USED = 21, S_ERR_EVENTS = 21 };

__device__ __forceinline__ ulonglong2 ld2(const u64* p) { return *reinterpret_cast<const ulonglong2*>(p); }
__device__ __forceinline__ void st2(u64* p, u64 a, u64 b) { *reinterpret_cast<ulonglong2*>(p) = make_ulonglong2(a, b); }

// ------------------------------------------------------------------------------------------------
// statistics: per-lane fold -> warp REDUX -> shared -> one global atomic per counter per CTA.  All
// threads of the CTA must call this (converged).  Tarok.rezultati accumulation (Tarok.py:59-61) is
// the S_PLAYER block: seat s of game i is player (s + i) % 4 (Tarok.py:34).
// ------------------------------------------------------------------------------------------------
struct GameStat { bool fin, err; u64 packed; u32 contract, plays; u64 gid; };

__device__ __forceinline__ u64 rotl64(u64 x, u32 r) { return r ? (x << r) | (x >> (64u - r)) : x; }

template <int NG>
__device__ __forceinline__ void accumulate_stats(long long* __restrict__ stats, const GameStat (&gs)[NG]) {
    __shared__ int sh[S_USED];                         // a CTA's sums fit 32 bits (<= 512 games x |score| <= 135, x 48 plays)
    if (threadIdx.x < S_USED) sh[threadIdx.x] = 0;
    __syncthreads();
    const unsigned full = 0xFFFFFFFFu;
    int sc[4] = {0, 0, 0, 0}, pl[4] = {0, 0, 0, 0}, steps = 0;
    // contract histogram: a warp holds at most 32 * NG <= 64 games, so one byte per contract cannot overflow when the
    // three words (contracts 0-3, 4-7, 8-9) are summed over the warp with REDUX
    u32 hist[3] = {0, 0, 0}, nfin = 0, nerr = 0;
#pragma unroll
    for (int k = 0; k < NG; k++) {
        const u64 by_seat = gs[k].fin ? gs[k].packed : 0ull;
        // seat s of game i is player (s + i) % 4: the scores by player are the seat scores rotated by 16 * (i % 4) bits
        const u64 by_player = rotl64(by_seat, 16u * ((u32)gs[k].gid & 3u));
#pragma unroll
        for (int s = 0; s < 4; s++) {
            sc[s] += (int)(int16_t)(by_seat >> (16 * s));
            pl[s] += (int)(int16_t)(by_player >> (16 * s));
        }
        steps += (int)gs[k].plays;
        const u32 c = gs[k].contract;
        const u32 inc = (gs[k].fin && c < 10u) ? 1u << (8u * (c & 3u)) : 0u;
        hist[0] += (c >> 2) == 0u ? inc : 0u; hist[1] += (c >> 2) == 1u ? inc : 0u; hist[2] += (c >> 2) == 2u ? inc : 0u;
        nfin += gs[k].fin ? 1u : 0u;
        nerr += gs[k].err ? 1u : 0u;
    }
    int mine = 0;
    const u32 lane = threadIdx.x & 31u;
#pragma unroll
    for (int s = 0; s < 4; s++) {
        int a = __reduce_add_sync(full, sc[s]);
        int b = __reduce_add_sync(full, pl[s]);
        if (lane == (u32)(S_SEAT + s)) mine = a;
        if (lane == (u32)(S_PLAYER + s)) mine = b;
    }
    {
        const u32 h0 = __reduce_add_sync(full, hist[0]), h1 = __reduce_add_sync(full, hist[1]), h2 = __reduce_add_sync(full, hist[2]);
        if (lane >= (u32)S_CONTRACT && lane < (u32)S_CONTRACT + 10u) {
            const u32 c = lane - (u32)S_CONTRACT;
            const u32 w = c < 4u ? h0 : c < 8u ? h1 : h2;
            mine = (int)((w >> (8u * (c & 3u))) & 255u);
        }
        const u32 a = __reduce_add_sync(full, nfin | (nerr << 16));
        const int b = __reduce_add_sync(full, steps);
        if (lane == S_FINISHED) mine = (int)(a & 0xFFFFu);
        if (lane == S_STEPS) mine = b;
        if (lane == S_ERRORS) mine = (int)(a >> 16);
    }
    if (lane < S_USED && mine != 0) atomicAdd(&sh[lane], mine);
    __syncthreads();
    if (threadIdx.x < S_USED && sh[threadIdx.x] != 0)
        atomicAdd((unsigned long long*)&stats[threadIdx.x], (unsigned long long)(long long)sh[threadIdx.x]);
}

// ------------------------------------------------------------------------------------------------
// deal: Igra.razdeli (Igra.py:65-73) with a counter-based Philox generator.
// Card c goes to a uniformly random free slot among the 54-c left = a walk over the remaining pile
// capacities (12,12,12,12,6); the talon ORDER is a uniform permutation decoded from one more draw.
// 55 bounded draws = 7 Philox blocks per deal (16-bit lanes): ALU-bound, not HBM-bound (DESIGN.md).
// ------------------------------------------------------------------------------------------------
struct Dealt { u64 h0, h1, h2, h3, talon, order; };

// ---- hand slots -------------------------------------------------------------------------------------------------
// hands[j * n_alloc + g] holds the hand of seat (leader + j) & 3, where leader is the M_LEADER field of the game's meta
// word (the seat that opens the current trick; 0 from the deal until a contract or a trick says otherwise).  The seat to
// move is therefore always in slot `pos`, the same slot for every game of a lock-step batch: play_step reads and writes
// ONE coalesced slot (plus the next seat's for its legal mask) instead of gathering from four seat-indexed arrays and
// scattering 8-byte writes; when a trick ends the four hands are re-written rotated to the winner.  Everything that
// changes the leader goes through these helpers.  tarok_hands_by_seat / TarokEnv.hands give the seat-indexed view.
__device__ __forceinline__ void rotate4(u64& a, u64& b, u64& c, u64& d, u32 r) {        // out[j] = in[(j + r) & 3]
    const bool by1 = r & 1u, by2 = r & 2u;                 // two conditional stages: by one, then by two
    const u64 a1 = by1 ? b : a, b1 = by1 ? c : b, c1 = by1 ? d : c, d1 = by1 ? a : d;
    a = by2 ? c1 : a1; b = by2 ? d1 : b1; c = by2 ? a1 : c1; d = by2 ? b1 : d1;
}
__device__ __forceinline__ void seats_to_slots(u64& a, u64& b, u64& c, u64& d, u32 leader) { rotate4(a, b, c, d, leader & 3u); }
__device__ __forceinline__ void slots_to_seats(u64& a, u64& b, u64& c, u64& d, u32 leader) { rotate4(a, b, c, d, (4u - leader) & 3u); }
__device__ __forceinline__ u32 slot_of(u32 seat, u32 leader) { return (seat - leader) & 3u; }
__device__ __forceinline__ u32 leader_of(u64 meta) { return ((u32)meta >> M_LEADER) & 3u; }

// Talon order = the L-th permutation (L < 720, Lehmer code, digits 120 / 24 / 6 / 2 / 1) of the six talon ids ascending:
// order field i = the d_i-th smallest id not taken yet.  All on 32-bit words: the permutation is decoded on the RANKS 0..5 kept
// as 4-bit fields of one register (a pick = one field extract + one masked merge), the ids are laid out one per byte in two
// registers, and one byte permute per output word maps ranks to ids (the rank nibbles are the permute's selectors).
// Equal to the 64-bit restatement (six ffs, Lehmer decode on a 36-bit packed list) for every L and talon
// (tests/test_setup_and_closer_exact.py).
__device__ __forceinline__ u64 order_from_lehmer(u64 talon, u32 L) {
    // Lehmer digits by constant multiplies, exact on the ranges they see (L < 720, r1 < 120, r2 < 24)
    const u32 d0 = (L * 1093u) >> 17, r1 = L - 120u * d0;
    const u32 d1 = (r1 * 2731u) >> 16, r2 = r1 - 24u * d1;
    const u32 d2 = (r2 * 43u) >> 8, r3 = r2 - 6u * d2;
    const u32 d3 = r3 >> 1, d4 = r3 & 1u;
    u32 rank = 0x543210u, perm = 0;                // ranks not taken yet, 4 bits each, ascending
    auto pick = [&](u32 d, int i) {
        const u32 sh = 4u * d;
        perm |= ((rank >> sh) & 15u) << (4 * i);
        const u32 high = 0xFFFFFFFFu << sh;        // fields d.. move down by one, fields below d stay
        rank = (rank & ~high) | ((rank >> 4) & high);
    };
    pick(d0, 0); pick(d1, 1); pick(d2, 2); pick(d3, 3); pick(d4, 4);
    perm |= rank << 20;                            // the one left
    // the six ids ascending, one per byte: bytes 0-3 in a, 4-5 in b (lowest set bit, then clear it, on the 32-bit halves)
    u32 lo = (u32)talon, hi = (u32)(talon >> 32), a = 0, b = 0;
#pragma unroll
    for (int i = 0; i < 6; i++) {
        const bool inlo = lo != 0u;
        const u32 w = inlo ? lo : hi;
        const u32 c = (u32)__ffs(w) - 1u + (inlo ? 0u : 32u);
        if (i < 4) a |= c << (8 * i); else b |= c << (8 * (i - 4));
        if (inlo) lo &= lo - 1u; else hi &= hi - 1u;
    }
    const u32 x = __byte_perm(a, b, perm & 0xFFFFu), y = __byte_perm(a, b, perm >> 16);   // ids in order, one per byte
    // bytes -> 6-bit fields
    const u32 olo = (x & 0x3Fu) | ((x >> 2) & 0xFC0u) | ((x >> 4) & 0x3F000u) | ((x >> 6) & 0xFC0000u);
    const u32 ohi = (y & 0x3Fu) | ((y >> 2) & 0xFC0u);
    return (u64)olo | ((u64)ohi << 24);
}

// The 53 bounded draws of a deal (n = 54 - c for card c; card 53 has no choice left) are BATCHED: several exact draws
// from one 32-bit Philox word (philox.cuh, bdraw): words 0..5 carry three cards each (cards 0..17), words 6..13 four each
// (cards 18..49), word 14 cards 50..52, word 15 whole the talon order (32-bit Lemire, n = 720).  16 words = 4 Philox
// blocks per deal (the 16-bit-lane version of round 1 needed 7), two multiplies per draw on the FMA pipe and one
// rejection compare per WORD (probability of a redraw < 1e-3 per deal; redraws go to stream ST_DEAL_RETRY).
// Card c lives in the low word of a bitboard for c < 32 and in the high word otherwise, which is known at
// compile time in the unrolled loop.
enum : u32 { ST_DEAL_RETRY = 7 };

__host__ __device__ constexpr int deal_first_card(int w) { return w < 6 ? 3 * w : w < 14 ? 18 + 4 * (w - 6) : 50; }
__host__ __device__ constexpr int deal_cards_in(int w) { return (w < 6 || w == 14) ? 3 : 4; }
__host__ __device__ constexpr u32 deal_prod(int w) {
    u32 p = 1;
    for (int i = 0; i < deal_cards_in(w); i++) p *= (u32)(54 - (deal_first_card(w) + i));
    return p;
}
__host__ __device__ constexpr u64 deal_bounds8(int w) {
    u64 b = 0;
    for (int i = 0; i < deal_cards_in(w); i++) b |= (u64)(54 - (deal_first_card(w) + i)) << (8 * i);
    return b;
}

// The pile walk keeps CUMULATIVE state: T_j = free slots in piles 0..j.  A draw r picks pile s = min{j : r < T_j}, i.e.
// q_j = (r < T_j) holds exactly for j >= s, and the update is T_j -= q_j.  The four T_j (<= 54) live in the four bytes of
// ONE register with bit 7 of every byte set, so that a single subtraction compares all four at once (bit 7 of byte j of
// T - (r + 1) * 0x01010101 survives iff r < T_j; no borrow can cross a byte: every byte stays >= 0x80 - 54); the four q_j of
// eight consecutive cards are shifted into one accumulator (byte j = their eight q_j bits) and transposed into the cumulative
// bitboards H_j = cards in piles 0..j with byte permutes at the end: 5 integer instructions per card after the
// draw.  The hands are H_0, H_1^H_0, H_2^H_1, H_3^H_2 and the talon ALL54 ^ H_3.
struct DealWalk { u32 T, acc; u32 rev[7]; };

__device__ __forceinline__ void deal_place(DealWalk& d, int c, u32 r) {             // c is a compile-time constant at every call
    const u32 q = ((r * 0xFEFEFEFFu + d.T) >> 7) & 0x01010101u;                     // byte j = (r < T_j)
    d.T -= q;
    d.acc = d.acc * 2u + q;
    if ((c & 7) == 7) { d.rev[c >> 3] = __brev(d.acc); d.acc = 0; }                 // byte 3 - j: bit jj = q_j of card 8 * (c >> 3) + jj
}

template <int W>
__device__ __forceinline__ void deal_word(DealWalk& d, u32 x, const Rng& rng, u64 gid) {
    constexpr int C0 = deal_first_card(W), NC = deal_cards_in(W);
    constexpr u32 THRESH = (u32)((1ull << 32) % deal_prod(W));
    u32 r[NC];
#pragma unroll
    for (int i = 0; i < NC; i++) r[i] = bdraw(x, (u32)(54 - (C0 + i)));
    if (__builtin_expect(x < THRESH, 0)) {
        const u64 p = bdraw_retry(rng.seed, gid, ST_DEAL_RETRY, (u32)W, deal_bounds8(W), (u32)NC);
#pragma unroll
        for (int i = 0; i < NC; i++) r[i] = (u32)(p >> (6 * i)) & 63u;
    }
#pragma unroll
    for (int i = 0; i < NC; i++) deal_place(d, C0 + i, r[i]);
}

__device__ __forceinline__ Dealt deal_philox(const Rng& rng, u64 gid) {
    // T holds T_j - 1 (+ 0x80) per byte, so that the comparison is ONE multiply-add: T - r * 0x01010101 = T + r * 0xFEFEFEFF
    DealWalk d;
    d.T = (0x80808080u | 12u | (24u << 8) | (36u << 16) | (48u << 24)) - 0x01010101u;
    d.acc = 0;
    u32 L;
    {
        const Words4 b = philox_block(rng, gid, ST_DEAL, 0u);
        deal_word<0>(d, b.w[0], rng, gid); deal_word<1>(d, b.w[1], rng, gid);
        deal_word<2>(d, b.w[2], rng, gid); deal_word<3>(d, b.w[3], rng, gid);
    }
    {
        const Words4 b = philox_block(rng, gid, ST_DEAL, 1u);
        deal_word<4>(d, b.w[0], rng, gid); deal_word<5>(d, b.w[1], rng, gid);
        deal_word<6>(d, b.w[2], rng, gid); deal_word<7>(d, b.w[3], rng, gid);
    }
    {
        const Words4 b = philox_block(rng, gid, ST_DEAL, 2u);
        deal_word<8>(d, b.w[0], rng, gid); deal_word<9>(d, b.w[1], rng, gid);
        deal_word<10>(d, b.w[2], rng, gid); deal_word<11>(d, b.w[3], rng, gid);
    }
    {
        const Words4 b = philox_block(rng, gid, ST_DEAL, 3u);
        deal_word<12>(d, b.w[0], rng, gid); deal_word<13>(d, b.w[1], rng, gid);
        deal_word<14>(d, b.w[2], rng, gid);
        const u64 m = (u64)b.w[3] * 720u;                        // word 15 whole: the talon order
        L = (u32)(m >> 32);
        if (__builtin_expect((u32)m < 256u, 0)) L = draw_loop(rng.seed, gid, ST_DEAL_RETRY, 54u, 720u, 0u);   // 2^32 % 720 = 256
    }
    deal_place(d, 53, 0u);                                       // the last card takes the last free slot
    d.rev[6] = __brev(d.acc << 2);                               // cards 48..53 sit at bits 7..2 of the last accumulator
    const u32* rev = d.rev;
    // 4 x 4 byte transposes: H_j.lo = byte (3 - j) of rev[0..3], H_j.hi = byte (3 - j) of rev[4..6]
    u64 H[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const u32 k = 3u - (u32)j;                               // source byte
        const u32 lo01 = __byte_perm(rev[0], rev[1], k | ((4u + k) << 4));            // bytes: [rev0.k, rev1.k, x, x]
        const u32 lo23 = __byte_perm(rev[2], rev[3], k | ((4u + k) << 4));
        const u32 lo = __byte_perm(lo01, lo23, 0x5410);                               // [lo01.0, lo01.1, lo23.0, lo23.1]
        const u32 hi45 = __byte_perm(rev[4], rev[5], k | ((4u + k) << 4));
        const u32 hi6 = (rev[6] >> (8u * k)) & 0xFFu;
        const u32 hi = (hi45 & 0xFFFFu) | (hi6 << 16);
        H[j] = ((u64)hi << 32) | lo;
    }
    Dealt dd;
    dd.h0 = H[0]; dd.h1 = H[1] ^ H[0]; dd.h2 = H[2] ^ H[1]; dd.h3 = H[3] ^ H[2];
    dd.talon = ALL54 ^ H[3];
    dd.order = order_from_lehmer(dd.talon, L);
    return dd;
}

__global__ void __launch_bounds__(CTA, 4) k_deal(Env e) {
    u64 g = (u64)blockIdx.x * CTA + threadIdx.x;
    if (g >= e.n_alloc) return;
    const u64 na = e.n_alloc;
    Dealt d = {0, 0, 0, 0, 0, 0};
    u64 meta = meta_pad();
    if (g < e.n) { d = deal_philox(e.rng, e.first_gid + g); meta = meta_fresh(); }
    e.hands[g] = d.h0; e.hands[na + g] = d.h1; e.hands[2 * na + g] = d.h2; e.hands[3 * na + g] = d.h3;
    e.piles[g] = 0; e.piles[na + g] = 0; e.piles[2 * na + g] = 0; e.piles[3 * na + g] = 0;
    e.talon[g] = d.talon; e.torder[g] = d.order; e.meta[g] = meta; e.mask[g] = 0;
    if (e.hands0) { e.hands0[g] = d.h0; e.hands0[na + g] = d.h1; e.hands0[2 * na + g] = d.h2; e.hands0[3 * na + g] = d.h3; }
    if (e.discard) e.discard[g] = 0;
    e.dpts[g] = 0;
}

// Deal injection (Igra.shuffle patch, Igra.py:10,67): perm uint8 [n,54].  The CTA stages its
// 256 x 54 bytes through shared memory with 16-byte loads, then each lane folds its row to bitboards.
__device__ __forceinline__ Dealt deal_from_perm(const uint8_t* row, bool& ok) {
    Dealt d = {0, 0, 0, 0, 0, 0};
    u64 seen = 0;
#pragma unroll
    for (int i = 0; i < 54; i++) {
        u32 c = row[i];
        u64 bit = c < 54 ? 1ull << c : 0ull;
        seen |= bit;
        if (i < 12) d.h0 |= bit; else if (i < 24) d.h1 |= bit; else if (i < 36) d.h2 |= bit;
        else if (i < 48) d.h3 |= bit; else { d.talon |= bit; d.order |= (u64)(c & 63u) << (6 * (i - 48)); }
    }
    ok = seen == ALL54;
    return d;
}

__global__ void __launch_bounds__(CTA) k_set_deals(Env e, const uint8_t* __restrict__ perm) {
    __shared__ __align__(16) uint8_t sh[CTA * 54];
    const u64 base = (u64)blockIdx.x * CTA;
    const u64 na = e.n_alloc;
    {   // CTA * 54 bytes = 864 x 16 B; rows past n are not read
        const u64 total = e.n * 54ull, off = base * 54ull;
        const bool vec_ok = (((uintptr_t)perm) & 15u) == 0;
        for (u32 v = threadIdx.x; v < CTA * 54 / 16; v += CTA) {
            u64 b = off + (u64)v * 16;
            if (vec_ok && b + 16 <= total) {
                *reinterpret_cast<uint4*>(sh + v * 16) = *reinterpret_cast<const uint4*>(perm + b);
            } else {
                for (int k = 0; k < 16; k++) sh[v * 16 + k] = (b + k < total) ? perm[b + k] : 0xFF;
            }
        }
    }
    __syncthreads();
    u64 g = base + threadIdx.x;
    if (g >= na) return;
    Dealt d = {0, 0, 0, 0, 0, 0};
    u64 meta = meta_pad();
    if (g < e.n) {
        bool ok;
        d = deal_from_perm(sh + threadIdx.x * 54, ok);
        meta = meta_fresh();
        if (!ok) { meta = mset(meta, M_PHASE, 2, PH_DONE) | (1ull << M_ERR); atomicAdd((unsigned long long*)&e.stats[S_ERR_EVENTS], 1ull); }
    }
    e.hands[g] = d.h0; e.hands[na + g] = d.h1; e.hands[2 * na + g] = d.h2; e.hands[3 * na + g] = d.h3;
    e.piles[g] = 0; e.piles[na + g] = 0; e.piles[2 * na + g] = 0; e.piles[3 * na + g] = 0;
    e.talon[g] = d.talon; e.torder[g] = d.order; e.meta[g] = meta; e.mask[g] = 0;
    if (e.hands0) { e.hands0[g] = d.h0; e.hands0[na + g] = d.h1; e.hands0[2 * na + g] = d.h2; e.hands0[3 * na + g] = d.h3; }
    if (e.discard) e.discard[g] = 0;
    e.dpts[g] = 0;
}

// Compact deal record (20 B = five u32 words; include/tarok_b200.h "deal records"): two bit planes over the 54 card ids
// give the seat of every hand card; the 45-bit word m -- the six talon ids in talon order (= `torder` as it stands) and the
// forced contract -- sits in the ten spare bits of each plane word and the fifth u32.  Decoding is a handful of bitwise
// ops plus six shifts for the talon set.
struct DealRecord { u32 contract, declarer, king; };
constexpr int RECORD_BYTES = 20;
__device__ __forceinline__ Dealt deal_from_record(const u32* a, DealRecord& r, bool& ok) {
    const u64 w0 = (u64)a[0] | ((u64)a[1] << 32), w1 = (u64)a[2] | ((u64)a[3] << 32);
    const u64 m = (w0 >> 54) | ((w1 >> 54) << 10) | ((u64)a[4] << 20);
    const u64 p0 = w0 & ALL54, p1 = w1 & ALL54;
    Dealt d;
    d.order = m & ((1ull << 36) - 1ull);
    u64 t = 0;
    u32 top = 0;
#pragma unroll
    for (int i = 0; i < 6; i++) {
        const u32 c = (u32)(d.order >> (6 * i)) & 63u;
        top = max(top, c);
        t |= 1ull << c;
    }
    d.talon = t;
    d.h0 = ALL54 & ~(p0 | p1 | t); d.h1 = p0 & ~p1; d.h2 = p1 & ~p0; d.h3 = p0 & p1;
    // two planes partition the ids into four classes; (12,12,12,12) + six distinct talon ids outside classes 1-3 <=> a deal
    ok = top < 54u && !(t & (p0 | p1)) && __popcll(t) == 6 && __popcll(d.h0) == 12 && __popcll(d.h1) == 12
         && __popcll(d.h2) == 12 && __popcll(d.h3) == 12 && (m >> 45) == 0ull;
    r.contract = (u32)(m >> 36) & 15u; r.declarer = (u32)(m >> 40) & 3u; r.king = (u32)(m >> 42) & 7u;
    return d;
}

// Current deal -> the permutation Igra.razdeli would have consumed (hands ascending, ordered talon).
__global__ void __launch_bounds__(CTA) k_export_perm(Env e, uint8_t* __restrict__ out) {
    __shared__ uint8_t sh[CTA * 54];
    const u64 base = (u64)blockIdx.x * CTA;
    u64 g = base + threadIdx.x;
    if (g < e.n) {
        uint8_t* row = sh + threadIdx.x * 54;
        const u64 na = e.n_alloc;
        int k = 0;
        const u32 leader = leader_of(e.meta[g]);
        for (int s = 0; s < 4; s++) {
            u64 h = e.hands[slot_of((u32)s, leader) * na + g];
            for (int i = 0; i < 12; i++) {
                u32 c = h ? (u32)__ffsll((long long)h) - 1u : 0xFFu;
                h &= h - 1;
                row[k++] = (uint8_t)c;
            }
        }
        u64 o = e.torder[g];
        for (int i = 0; i < 6; i++) row[48 + i] = (uint8_t)((o >> (6 * i)) & 63ull);
    }
    __syncthreads();
    const u64 total = e.n * 54ull, off = base * 54ull;
    for (u32 b = threadIdx.x; b < CTA * 54; b += CTA)
        if (off + b < total) out[off + b] = sh[b];
}

// ------------------------------------------------------------------------------------------------
// contract start: auction (Igra.licitacija) or forced contract, then Igra.start dispatch + teams.
// ------------------------------------------------------------------------------------------------
// SRC_MIXED: per-seat players, fixed intents (a) beside Bot_igralec seats (bit s of the mask byte b[g]): tarok_auction_bots
enum : int { SRC_FORCED = 0, SRC_INTENTS = 1, SRC_SYNTH = 2, SRC_MIXED = 3 };

struct WantFixed { int tip[4]; __device__ int operator()(int seat, int) const {
    return seat == 0 ? tip[0] : seat == 1 ? tip[1] : seat == 2 ? tip[2] : tip[3]; }
    __device__ bool fixed(int) const { return true; } };
// np.random.choice([Naprej,Tri,Dve,Ena], p=[.5,1/6,1/6,1/6]) at EVERY call (Igralec.py:151): call i takes the i-th of the
// sixteen base-6 digits decoded from words 0 and 1 of the bid block (eight batched draws per word); an auction of
// Bot players never needs more (the bids only rise Tri -> Dve -> Ena), calls past 16 would use one word each.
struct WantBot { const Rng& rng; u64 gid; u64 digits; __device__ int operator()(int, int call) const {
    const u32 u = call < 16 ? (u32)(digits >> (3 * call)) & 7u : draw(rng, gid, ST_BID, 64u + (u32)call, 6u);
    return u < 3u ? (int)C_NAPREJ : (int)(C_TRI + (u - 3u)); }
    __device__ bool fixed(int) const { return false; } };
// Bot seats (bit s of `bots`) ask WantBot afresh at every call -- at overall call c the draw mode 18 takes at call c --, the
// other seats keep their fixed intent.
struct WantMixed { WantFixed f; WantBot b; u32 bots;
    __device__ bool fixed(int seat) const { return !((bots >> seat) & 1u); }
    __device__ int operator()(int seat, int call) const { return fixed(seat) ? f(seat, call) : b(seat, call); } };

constexpr u64 BOUNDS8_6x8 = 0x0606060606060606ull;
__device__ __forceinline__ u32 bot_digits8(u32 x, const Rng& rng, u64 gid, u32 word) {    // eight draws of [0,6) -> 3 bits each
    u32 out = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) out |= bdraw(x, 6u) << (3 * i);
    if (__builtin_expect(x < (u32)((1ull << 32) % 1679616ull), 0)) {
        const u64 p = bdraw_retry(rng.seed, gid, ST_BID, word, BOUNDS8_6x8, 8u);
        out = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) out |= ((u32)(p >> (6 * i)) & 7u) << (3 * i);
    }
    return out;
}

// The synthetic pre-play decisions of one game other than the bids come from ONE Philox block, (gid, ST_FORCE, 0):
//   word 0: forced contract of the mixed mode (n = 3), declarer (4), called king (4) -- three batched draws;
//   word 1: talon exchange -- the k discards (n = a, a-1, a-2 with a = discardable cards after the pick-up), batched;
//   word 2: the king a Bot_igralec declarer calls (n = 4, Igralec.py:155-156);
//   word 3: the talon group when it is random (n = number of groups, Igralec.py:369-370).
__device__ __forceinline__ Words4 setup_block(const Rng& rng, u64 gid) { return philox_block(rng, gid, ST_FORCE, 0u); }

// Resolves (contract, declarer, king) for one game from the chosen source.  `sb` = setup_block (SRC_SYNTH only).
template <int SRC>
__device__ __forceinline__ void resolve_contract(const Rng& rng, u64 gid, u32 mode, const uint8_t* a, const uint8_t* b,
                                                 const uint8_t* c, u64 g, const Words4& sb, u32& contract, u32& declarer,
                                                 u32& king) {
    if (SRC == SRC_FORCED) {
        contract = a[g]; declarer = b[g]; king = c ? c[g] : NO_KING;
    } else if (SRC == SRC_INTENTS) {
        uchar4 in = reinterpret_cast<const uchar4*>(a)[g];
        WantFixed w; u32 su[4];
        index2igra(in.x, w.tip[0], su[0]); index2igra(in.y, w.tip[1], su[1]);
        index2igra(in.z, w.tip[2], su[2]); index2igra(in.w, w.tip[3], su[3]);
        int d, k;
        licitacija(w, d, k);
        contract = (u32)k; declarer = (u32)d;
        // king = the suit attached to the declarer's ORIGINAL intent (Igralec.py:298,308-310)
        king = d == 0 ? su[0] : d == 1 ? su[1] : d == 2 ? su[2] : su[3];
        // every seat is asked at least once, so every intent counts: one past index 19 (index2igra[idx] would raise in
        // the reference) makes an error game through begin_contract's unknown-contract check
        if (max(max((u32)in.x, (u32)in.y), max((u32)in.z, (u32)in.w)) > 19u) contract = C_NONE;
    } else if (SRC == SRC_MIXED) {
        const uchar4 in = reinterpret_cast<const uchar4*>(a)[g];
        const u32 bots = b[g];
        // the bid block is only needed when a bot seat bids (words 0-1: sixteen base-6 digits, as in mode 18)
        u64 digits = 0;
        if (bots & 15u) {
            const Words4 bb = philox_block(rng, gid, ST_BID, 0u);
            digits = (u64)bot_digits8(bb.w[0], rng, gid, 0u) | ((u64)bot_digits8(bb.w[1], rng, gid, 1u) << 24);
        }
        WantMixed w{WantFixed{}, WantBot{rng, gid, digits}, bots};
        u32 su[4];
        index2igra(in.x, w.f.tip[0], su[0]); index2igra(in.y, w.f.tip[1], su[1]);
        index2igra(in.z, w.f.tip[2], su[2]); index2igra(in.w, w.f.tip[3], su[3]);
        int d, k;
        licitacija(w, d, k);
        contract = (u32)k; declarer = (u32)d;
        // a bot declarer of a king game calls the king of setup-block word 2 (as mode 18), a neural one the suit of its
        // original intent (as tarok_auction)
        const u32 sd = d == 0 ? su[0] : d == 1 ? su[1] : d == 2 ? su[2] : su[3];
        king = ((bots >> d) & 1u) ? (is_king_game(contract) ? draw(rng, gid, ST_FORCE, 2u, 4u) : NO_KING) : sd;
        // the intent of a bot seat is never read; one past index 19 at another seat, or a mask bit above seat 3, makes an
        // error game through begin_contract's unknown-contract check
        const u32 top = max(max((bots & 1u) ? 0u : (u32)in.x, (bots & 2u) ? 0u : (u32)in.y),
                            max((bots & 4u) ? 0u : (u32)in.z, (bots & 8u) ? 0u : (u32)in.w));
        if (top > 19u || bots > 15u) contract = C_NONE;
    } else {
        if (mode == 17u) {          // TAROK_MODE_AUCTION_UNIFORM: four batched draws of [0,18) from word 0 of the bid block
            u32 x = philox_block(rng, gid, ST_BID, 0u).w[0];
            u32 idx[4];
#pragma unroll
            for (int s = 0; s < 4; s++) idx[s] = bdraw(x, 18u);
            if (__builtin_expect(x < (u32)((1ull << 32) % 104976ull), 0)) {
                const u64 p = bdraw_retry(rng.seed, gid, ST_BID, 0u, 0x12121212ull, 4u);
#pragma unroll
                for (int s = 0; s < 4; s++) idx[s] = (u32)(p >> (6 * s)) & 63u;
            }
            WantFixed w; u32 su[4];
#pragma unroll
            for (int s = 0; s < 4; s++) index2igra(idx[s], w.tip[s], su[s]);
            int d, k;
            licitacija(w, d, k);
            contract = (u32)k; declarer = (u32)d;
            king = d == 0 ? su[0] : d == 1 ? su[1] : d == 2 ? su[2] : su[3];
        } else if (mode == 18u) {   // TAROK_MODE_AUCTION_BOT
            const Words4 bb = philox_block(rng, gid, ST_BID, 0u);
            WantBot w{rng, gid, (u64)bot_digits8(bb.w[0], rng, gid, 0u) | ((u64)bot_digits8(bb.w[1], rng, gid, 1u) << 24)};
            int d, k;
            licitacija(w, d, k);
            contract = (u32)k; declarer = (u32)d;
            king = is_king_game(contract) ? draw_from_word(sb.w[2], rng, gid, ST_FORCE, 2u, 4u) : NO_KING;   // Igralec.py:155-156
        } else {
            u32 x = sb.w[0];
            u32 c3 = bdraw(x, 3u), d4 = bdraw(x, 4u), k4 = bdraw(x, 4u);
            if (__builtin_expect(x < 16u, 0)) {                                  // 2^32 mod 48
                const u64 p = bdraw_retry(rng.seed, gid, ST_FORCE, 0u, 0x040403ull, 3u);
                c3 = (u32)p & 63u; d4 = (u32)(p >> 6) & 63u; k4 = (u32)(p >> 12) & 63u;
            }
            contract = mode == 16u ? C_TRI + c3 : mode;
            declarer = contract == C_KLOP ? 0u : d4;
            king = is_king_game(contract) ? k4 : NO_KING;
        }
    }
}

template <int SRC>
__global__ void __launch_bounds__(CTA) k_begin(Env e, u32 mode, const uint8_t* __restrict__ a,
                                               const uint8_t* __restrict__ b, const uint8_t* __restrict__ c) {
    u64 g = (u64)blockIdx.x * CTA + threadIdx.x;
    if (g >= e.n) return;
    u64 meta = e.meta[g];
    if (mget(meta, M_PHASE, 2) != PH_DEALT || ((meta >> M_ERR) & 1ull)) return;
    const u64 na = e.n_alloc;
    u64 h0 = e.hands[g], h1 = e.hands[na + g], h2 = e.hands[2 * na + g], h3 = e.hands[3 * na + g];
    u32 contract, declarer, king;
    Words4 sb = {{0, 0, 0, 0}};
    const u64 gid = e.first_gid + g;
    if (SRC == SRC_SYNTH) sb = setup_block(e.rng, gid);
    resolve_contract<SRC>(e.rng, gid, mode, a, b, c, g, sb, contract, declarer, king);
    slots_to_seats(h0, h1, h2, h3, leader_of(meta));             // identity in practice: a dealt game has leader 0
    meta = begin_contract(meta, contract, declarer, king, h0, h1, h2, h3);
    if ((meta >> M_ERR) & 1ull) atomicAdd((unsigned long long*)&e.stats[S_ERR_EVENTS], 1ull);
    e.meta[g] = meta;
    e.mask[g] = mask_for_mover(meta, sel4(h0, h1, h2, h3, mover_of(meta)));
    if (leader_of(meta) != 0u) {                                  // Berac: the declarer opens -> re-seat the slots
        seats_to_slots(h0, h1, h2, h3, leader_of(meta));
        e.hands[g] = h0; e.hands[na + g] = h1; e.hands[2 * na + g] = h2; e.hands[3 * na + g] = h3;
    }
}

// ------------------------------------------------------------------------------------------------
// talon exchange: Navadna_igra.odpri_talon/start (Navadna_igra.py:36-68); the declarer takes group g
// and lays k discardable cards (Roka.mozno_zalozit, Roka.py:23-27) into the own pile (Igralec.py:161-171).
// ------------------------------------------------------------------------------------------------
// Returns false (error) if the action is invalid or fewer than k cards can be laid down (Q19).
// SYNTH: the decision is drawn from words 1 and 3 of the setup block `sb`.
// Card points of a bitboard (Roka.vrednost_stiha's per-card values, Roka.py:76-91): 1 + J 1, C 2, Q 3, K / trula 4 extra.
__device__ __forceinline__ u32 card_points(u64 s) {
    return (u32)(__popcll(s) + __popcll(s & JACKS) + 2 * __popcll(s & CAVALS) + 3 * __popcll(s & QUEENS)
                 + 4 * __popcll(s & (KINGS | TRULA)));
}

// sel8: the byte-select table in shared memory (select8_to_shared) for the discard picks, or nullptr in kernels that have none
// (the binary descent then runs to the end); both give the same card.
template <bool SYNTH>
__device__ __forceinline__ bool exchange_game(const Rng& rng, u64 gid, u32 random_group, const Words4& sb, u64& meta, u64& hand,
                                              u64& pile, u64& talon, u64 order, u32 group, u64 discard, u64& discard_out,
                                              const uint8_t* __restrict__ sel8 = nullptr) {
    u32 contract = mget(meta, M_CONTRACT, 4);
    u32 k = talon_k(contract);
    u32 ngroups = 6u / k;
    u64 gb_synth = 0;
    if (SYNTH) {
        // Bot: group 0 (Igralec.py:162); neural random branch: a uniform group (Igralec.py:369-370), its own word
        group = random_group ? draw_from_word(sb.w[3], rng, gid, ST_FORCE, 3u, ngroups) : 0u;
        gb_synth = talon_group_bits(order, k, group);
        u64 avail = (hand | gb_synth) & DISCARDABLE;
        const u32 a = (u32)__popcll(avail);
        if (a < k) return false;
        u32 x = sb.w[1], prod = 1, rd[3] = {0, 0, 0};
#pragma unroll
        for (u32 j = 0; j < 3; j++) if (j < k) { rd[j] = bdraw(x, a - j); prod *= a - j; }
        if (__builtin_expect(x < prod, 0) && x < (0u - prod) % prod) {           // rejected sliver: redraw the word
            u64 bb = 0;
            for (u32 j = 0; j < k; j++) bb |= (u64)(a - j) << (8 * j);
            const u64 p1 = bdraw_retry(rng.seed, gid, ST_FORCE, 1u, bb, k);
            for (u32 j = 0; j < 3; j++) rd[j] = (u32)(p1 >> (6 * j)) & 63u;
        }
        discard = 0;
#pragma unroll
        for (u32 j = 0; j < 3; j++) if (j < k) {    // uniform k-subset = random.sample (Igralec.py:166)
            u64 bit = 1ull << (sel8 ? nth_set_bit_lut(avail, rd[j], sel8) : nth_set_bit(avail, rd[j]));
            avail ^= bit; discard |= bit;
        }
    }
    if (group >= ngroups) return false;
    const u64 gb = SYNTH ? gb_synth : talon_group_bits(order, k, group);
    u64 full = hand | gb;
    if ((u32)__popcll(discard) != k || (discard & ~(full & DISCARDABLE))) return false;
    hand = full & ~discard;
    pile |= discard;
    talon &= ~gb;
    discard_out = discard;
    meta = mset(meta, M_GROUP, 3, group);
    meta = mset(meta, M_PHASE, 2, PH_PLAY);
    return true;
}

// BOTS (tarok_exchange_bots): a game whose declarer's seat has its bit set in bots[g] takes the synthetic Bot exchange
// (group 0, the discards of setup-block word 1) and ignores its group / discard entries; a mask byte above 15 is an error.
template <bool SYNTH, bool BOTS = false>
__global__ void __launch_bounds__(CTA) k_exchange(Env e, u32 random_group, const uint8_t* __restrict__ group,
                                                  const u64* __restrict__ discard, const uint8_t* __restrict__ bots) {
    u64 g = (u64)blockIdx.x * CTA + threadIdx.x;
    if (g >= e.n) return;
    u64 meta = e.meta[g];
    if (mget(meta, M_PHASE, 2) != PH_EXCHANGE) return;
    const u64 na = e.n_alloc;
    u32 decl = mget(meta, M_DECL, 2);
    u64 h0 = e.hands[g], h1 = e.hands[na + g], h2 = e.hands[2 * na + g], h3 = e.hands[3 * na + g];
    const u32 leader = leader_of(meta);
    slots_to_seats(h0, h1, h2, h3, leader);
    u64 hand = sel4(h0, h1, h2, h3, decl);
    u64 pile = e.piles[decl * na + g];
    u64 talon = e.talon[g], order = e.torder[g], dout = 0;
    Words4 sb = {{0, 0, 0, 0}};
    const u64 gid = e.first_gid + g;
    const u32 bm = BOTS ? (u32)bots[g] : 0u;
    const bool bot = BOTS && ((bm >> decl) & 1u);
    if (SYNTH || bot) sb = setup_block(e.rng, gid);
    bool ok;
    if (BOTS && bm > 15u) ok = false;
    else if (bot) ok = exchange_game<true>(e.rng, gid, 0u, sb, meta, hand, pile, talon, order, 0u, 0ull, dout);
    else ok = exchange_game<SYNTH>(e.rng, gid, random_group, sb, meta, hand, pile, talon, order,
                                   SYNTH ? 0u : (u32)group[g], SYNTH ? 0ull : discard[g], dout);
    if (!ok) {
        meta = mset(meta, M_PHASE, 2, PH_DONE) | (1ull << M_ERR);
        atomicAdd((unsigned long long*)&e.stats[S_ERR_EVENTS], 1ull);
        e.meta[g] = meta;
        e.mask[g] = 0;
        return;
    }
    e.hands[slot_of(decl, leader) * na + g] = hand;
    e.piles[decl * na + g] = pile;
    e.talon[g] = talon;
    e.meta[g] = meta;
    if (e.discard) e.discard[g] = dout;
    e.dpts[g] = (uint8_t)card_points(dout);
    u32 mv = mover_of(meta);
    e.mask[g] = mask_for_mover(meta, mv == decl ? hand : sel4(h0, h1, h2, h3, mv));
}

// ------------------------------------------------------------------------------------------------
// play_step: one card per live game per launch -- THE hot kernel (48 launches per deal).
// Algorithmic traffic per env-step (SURVEY.md 8d): R meta 8 + hands 16 + action 1, W hand 8 + meta 8
// + mask 8, per trick /4: pile RW 16 (+ Klop talon) = 64 B.  What a lock-step batch moves: R meta 8 + the mover's and
// the next seat's slot 16, W slot 8 + meta 8 + mask 8; the trick-closing step reads and re-writes all four slots
// (rotation to the winner) and appends a 4-byte trick-log entry: 59 B on average.
// ------------------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------------------
// setup: deal -> contract (synthetic mode) -> talon exchange fused into ONE launch for pipelines whose
// pre-play decisions are all made on the device (uniform-random / Bot players).  Same device functions and
// Philox draws as k_deal + k_begin<SYNTH> + k_exchange<SYNTH>, so the resulting state is bit-identical; the
// state is written once instead of written, re-read and patched twice.
// ------------------------------------------------------------------------------------------------
template <bool GRAPH = false>
__global__ void __launch_bounds__(CTA, TK_SETUP_BLOCKS) k_setup_synth(Env e, u32 mode) {
    __shared__ __align__(16) uint8_t sel8[SELECT8_SMEM];  // byte-select table of the discard picks (tarok_rules.cuh)
    select8_to_shared(sel8);
    if constexpr (GRAPH) load_run_params(e);
    __syncthreads();                                      // every lane reaches this: the grid covers n_alloc exactly
    const u64 g = (u64)blockIdx.x * CTA + threadIdx.x;
    const u64 na = e.n_alloc;
    if (g >= na) return;
    Dealt d = {0, 0, 0, 0, 0, 0};
    u64 meta = meta_pad(), mask = 0, dout = 0, hand = 0;
    u32 decl = 0;
    bool exchanged = false;
    if (g < e.n) {
        const u64 gid = e.first_gid + g;
        d = deal_philox(e.rng, gid);
        if (e.hands0) { e.hands0[g] = d.h0; e.hands0[na + g] = d.h1; e.hands0[2 * na + g] = d.h2; e.hands0[3 * na + g] = d.h3; }
        u32 contract, declarer, king;
        const Words4 sb = setup_block(e.rng, gid);
        resolve_contract<SRC_SYNTH>(e.rng, gid, mode, nullptr, nullptr, nullptr, g, sb, contract, declarer, king);
        meta = begin_contract(meta_fresh(), contract, declarer, king, d.h0, d.h1, d.h2, d.h3);
        decl = mget(meta, M_DECL, 2);
        if (mget(meta, M_PHASE, 2) == PH_EXCHANGE) {
            u64 pile = 0;
            hand = sel4(d.h0, d.h1, d.h2, d.h3, decl);
            exchanged = exchange_game<true>(e.rng, gid, mode == 17u, sb, meta, hand, pile, d.talon, d.order, 0u, 0ull, dout,
                                        sel8);
            if (!exchanged) meta = mset(meta, M_PHASE, 2, PH_DONE) | (1ull << M_ERR);
        }
        if ((meta >> M_ERR) & 1ull) atomicAdd((unsigned long long*)&e.stats[S_ERR_EVENTS], 1ull);
        // the opening seat's legal set; only Berac opens from another seat than 0, and then the four slots are re-seated
        const u32 leader = leader_of(meta);
        u64 opener = d.h0;
        if (leader != 0u) {
            opener = sel4(d.h0, d.h1, d.h2, d.h3, leader);
            seats_to_slots(d.h0, d.h1, d.h2, d.h3, leader);
        }
        if (exchanged && decl == leader) opener = hand;
        mask = mask_for_mover(meta, opener);
    } else if (e.hands0) {
        e.hands0[g] = 0; e.hands0[na + g] = 0; e.hands0[2 * na + g] = 0; e.hands0[3 * na + g] = 0;
    }
    // the hands as dealt (leader-relative), empty piles; an exchange then overwrites the declarer's two words -- the
    // contracts that exchange all open from seat 0, so the declarer's slot is its seat
    e.hands[g] = d.h0; e.hands[na + g] = d.h1; e.hands[2 * na + g] = d.h2; e.hands[3 * na + g] = d.h3;
    e.piles[g] = 0; e.piles[na + g] = 0; e.piles[2 * na + g] = 0; e.piles[3 * na + g] = 0;
    if (exchanged) { e.hands[decl * na + g] = hand; e.piles[decl * na + g] = dout; }
    e.talon[g] = d.talon; e.torder[g] = d.order; e.meta[g] = meta; e.mask[g] = mask;
    if (e.discard) e.discard[g] = dout;
    e.dpts[g] = (uint8_t)card_points(dout);
}

// TAROK_CARD_SKIP (0xFE) as the supplied card leaves a live game untouched for this launch (a caller that advances only a
// subset of the live games, e.g. the Solo_brez one-step lead of the reference's lock-step scheduler, SURVEY Q17).
constexpr u32 CARD_SKIP = 0xFEu;
// The two card ids of a lane's game pair.  The caller's array holds exactly n_games bytes: never read past it.
__device__ __forceinline__ u32 load_actions(const uint8_t* __restrict__ action, u32 g, u64 n) {
    if ((u64)g + 1 < n) return *reinterpret_cast<const unsigned short*>(action + g);
    return (u64)g < n ? (u32)action[g] | 0xFF00u : 0xFFFFu;
}

// Programmatic dependent launch (PDL): consecutive play_step launches are chained so that the CTAs of step
// t+1 are scheduled while the tail of step t drains; they park at griddepcontrol.wait until step t has
// completed and its writes are visible.  This removes the launch ramp / tail bubble between the 48 steps.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// Game indices are 32-bit inside the step kernels (n_alloc <= 2^29, enforced by tarok_create): one IMAD.WIDE
// per address instead of 64-bit multiply chains.

// The masks of a game pair after a step.  A live game that was told to skip (CARD_SKIP) keeps the mask it has; that
// can only happen with externally supplied cards, and then the pair is written with scalar stores.
// MASK = false (interior launches of a chain of in-kernel random steps, whose masks nobody can observe): nothing is
// computed or stored, except that a game FINISHING in this launch gets its mask cleared -- no later launch touches it.
template <bool RANDOM, bool MASK>
__device__ __forceinline__ void store_masks(const Env& e, u32 g, const ulonglong2& m, bool a0, bool a1, u64 k0, u64 k1) {
    if (!MASK) {
        if (a0 && (((u32)m.x >> M_PHASE) & 3u) != PH_PLAY) e.mask[g] = 0ull;
        if (a1 && (((u32)m.y >> M_PHASE) & 3u) != PH_PLAY) e.mask[g + 1] = 0ull;
        return;
    }
    const bool sk0 = !RANDOM && !a0 && (((u32)m.x >> M_PHASE) & 3u) == PH_PLAY && !((m.x >> M_ERR) & 1ull),
               sk1 = !RANDOM && !a1 && (((u32)m.y >> M_PHASE) & 3u) == PH_PLAY && !((m.y >> M_ERR) & 1ull);
    if (!sk0 && !sk1) { st2(e.mask + g, k0, k1); return; }
    if (!sk0) e.mask[g] = k0;
    if (!sk1) e.mask[g + 1] = k1;
}

// ---- action sources of play_step: RANDOM = in-kernel uniform-random players (tarok_step_random); otherwise the caller's
// card bytes (tarok_step), and with BOTS (tarok_step_bots) the per-game seat mask `bm` (bit s = seat s is a Bot_igralec):
// a bot mover plays the uniform legal card tarok_step_random would play at that play index (play_draw on (gid, plays)) and
// its card byte is ignored, except CARD_SKIP, which holds the game as for everybody.  A mask byte above 15 makes the game an
// error game (counted at once, like an illegal card).
__device__ __forceinline__ bool bot_moves(u64 meta, u32 bm) { return (bm >> mover_of(meta)) & 1u; }
__device__ __forceinline__ u64 input_error(const Env& e, u64 meta) {
    atomicAdd((unsigned long long*)&e.stats[S_ERR_EVENTS], 1ull);
    return mset(meta, M_PHASE, 2, PH_DONE) | (1ull << M_ERR);
}

// ---- general path: any mix of trick positions; the four slots of the game are in registers ----------------------
template <bool RANDOM, bool MASK, bool BOTS = false>
__device__ __forceinline__ void step_game_any(const Env& e, u32 g, u64& meta, u64 s0, u64 s1, u64 s2, u64 s3, u32 card,
                                              const Words4& rnd, u64& next_mask, u32 bm = 0u) {
    const u32 na = (u32)e.n_alloc;
    const u32 lo = (u32)meta, hi = (u32)(meta >> 32);
    const u32 pos = (lo >> M_POS) & 3u, leader = (lo >> M_LEADER) & 3u, kf = (lo >> M_KLOPFAM) & 1u;
    const u32 mover = (leader + pos) & 3u;
    const u32 plays = (hi >> (M_PLAYS - 32)) & 63u;
    u64 hand = sel4(s0, s1, s2, s3, pos);                          // the seat to move sits in slot `pos`
    if (BOTS && bm > 15u) { meta = input_error(e, meta); next_mask = 0; return; }
    if (RANDOM || (BOTS && ((bm >> mover) & 1u))) {
        const u64 legal = legal_moves(hand, pos != 0, hi & 63u, kf);
        card = nth_set_bit(legal, play_draw<-1>(rnd, e.rng, e.first_gid + g, plays, (u32)__popcll(legal)));
    }
    PlayResult pr;
    meta = play_card<!RANDOM, -1, false>(meta, hand, card, 0ull, 0ull, pr);
    next_mask = 0;
    if (!RANDOM && ((meta >> M_ERR) & 1ull)) {
        atomicAdd((unsigned long long*)&e.stats[S_ERR_EVENTS], 1ull);
        return;
    }
    if (e.hist) e.hist[(u64)plays * na + g] = (uint8_t)((mover << 6) | card);
    if (!pr.trick_done) {                                          // same trick goes on: next slot follows the same lead
        e.hands[pos * na + g] = hand;
        if (MASK) next_mask = legal_moves(sel4(s0, s1, s2, s3, (pos + 1u) & 3u), true, (u32)(meta >> 32) & 63u, kf);
    } else {
        // append-only trick log (4 B, coalesced) instead of a scattered read-modify-write of the winner's pile;
        // k_score materialises the piles (and the Klop talon) from it
        e.tricklog[(u64)(plays >> 2) * na + g] = log_entry((u32)(meta >> 32) & 0xFFFFFFu, pr.winner, (u32)meta);   // 12 rows: 64-bit index
        s3 = hand;                                                 // the trick closes from slot 3
        const u32 w = pr.winner_rel;                               // the winner's slot = its index in the trick
        if (w == 0u) {
            e.hands[3 * na + g] = s3;                              // the leader stays: only the mover's slot changed
        } else {
            rotate4(s0, s1, s2, s3, w);
            e.hands[g] = s0; e.hands[na + g] = s1; e.hands[2 * na + g] = s2; e.hands[3 * na + g] = s3;
        }
        if (MASK) next_mask = mask_for_mover(meta, s0);
    }
}

// Philox block(s) for the two games of a lane: one block serves both (same pair, same trick) in the common case.
__device__ __forceinline__ void pair_blocks(const Env& e, u32 g, u32 t0, u32 t1, bool a1, Words4& r0, Words4& r1) {
    const u64 gid = e.first_gid + g;
    r0 = play_block(e.rng, gid, t0);
    r1 = r0;
    if (((gid & 1ull) || t0 != t1) && a1) r1 = play_block(e.rng, gid + 1, t1);
}

template <bool RANDOM, bool MASK = true, bool BOTS = false>
__device__ __forceinline__ void step_pair_any(const Env& e, u32 g, ulonglong2& m, bool a0, bool a1, ulonglong2 s0,
                                              ulonglong2 s1, ulonglong2 s2, ulonglong2 s3, u32 act, u32 bm2 = 0u) {
    Words4 r0 = {{0, 0, 0, 0}}, r1 = {{0, 0, 0, 0}};
    const u32 t0 = ((u32)(m.x >> 32) >> (M_PLAYS - 30)) & 15u, t1 = ((u32)(m.y >> 32) >> (M_PLAYS - 30)) & 15u;
    if (RANDOM) pair_blocks(e, g, t0, t1, a1, r0, r1);
    if (BOTS) {                                                    // Philox only for a pair with a bot to move
        const bool b1 = a1 && bot_moves(m.y, bm2 >> 8);
        if ((a0 && bot_moves(m.x, bm2 & 0xFFu)) || b1) pair_blocks(e, g, t0, t1, b1, r0, r1);
    }
    u64 k0 = 0, k1 = 0;
    if (a0) step_game_any<RANDOM, MASK, BOTS>(e, g, m.x, s0.x, s1.x, s2.x, s3.x, act & 0xFFu, r0, k0, bm2 & 0xFFu);
    if (a1) step_game_any<RANDOM, MASK, BOTS>(e, g + 1, m.y, s0.y, s1.y, s2.y, s3.y, act >> 8, r1, k1, bm2 >> 8);
    st2(e.meta + g, m.x, m.y);
    store_masks<RANDOM, MASK>(e, g, m, a0, a1, k0, k1);
}

// General path for a lane pair.  HAVE = the trick position whose slots the caller has loaded already (a lock-step kernel
// whose warp vote failed: slot HAVE in `hm`, slot HAVE + 1 in `n0`, for HAVE == 3 also slots 1, 2 in `n1`, `n2`), or -1.
// Using them here also keeps those loads above the vote: one memory round trip on the lock-step side.
// MASK = false: the caller did not load the next seat's slot (n0) for HAVE < 3; it is fetched here.
template <bool RANDOM, int HAVE, bool MASK = true, bool BOTS = false>
__device__ __forceinline__ void step_pair_general(const Env& e, u32 g, ulonglong2 m, bool a0, bool a1, u32 act,
                                                  ulonglong2 hm, ulonglong2 n0, ulonglong2 n1, ulonglong2 n2, u32 bm2 = 0u) {
    const u32 na = (u32)e.n_alloc;
    ulonglong2 s0, s1, s2, s3;
    if (HAVE >= 0 && HAVE < 3 && !MASK) n0 = ld2(e.hands + ((HAVE + 1) * na + g));
    if (HAVE == 0) { s0 = hm; s1 = n0; s2 = ld2(e.hands + (2 * na + g)); s3 = ld2(e.hands + (3 * na + g)); }
    else if (HAVE == 1) { s1 = hm; s2 = n0; s0 = ld2(e.hands + g); s3 = ld2(e.hands + (3 * na + g)); }
    else if (HAVE == 2) { s2 = hm; s3 = n0; s0 = ld2(e.hands + g); s1 = ld2(e.hands + (na + g)); }
    else if (HAVE == 3) { s3 = hm; s0 = n0; s1 = n1; s2 = n2; }
    else { s0 = ld2(e.hands + g); s1 = ld2(e.hands + (na + g)); s2 = ld2(e.hands + (2 * na + g)); s3 = ld2(e.hands + (3 * na + g)); }
    step_pair_any<RANDOM, MASK, BOTS>(e, g, m, a0, a1, s0, s1, s2, s3, act, bm2);
}

// Cold paths of the lock-step kernels: the warp whose vote failed, and the draw-cache miss at trick positions 1-3.
// Inlined: out of line measured slower (profiles/r02/step_ab_run6.txt): 8.78 vs 7.98 us per launch at 1 M deals.
template <bool RANDOM, int HAVE, bool MASK, bool BOTS = false>
__device__ __forceinline__ void step_pair_general_cold(const Env& e, u32 g, ulonglong2 m, bool a0, bool a1, u32 act,
                                                    ulonglong2 hm, ulonglong2 n0, ulonglong2 n1, ulonglong2 n2, u32 bm2 = 0u) {
    step_pair_general<RANDOM, HAVE, MASK, BOTS>(e, g, m, a0, a1, act, hm, n0, n1, n2, bm2);
}
template <int POS>
__device__ __forceinline__ u32 pair_lanes_cold(const Env& e, u32 g, u32 trick, bool a1) {
    Words4 r0, r1;
    pair_blocks(e, g, trick, trick, a1, r0, r1);
    const u64 gid = e.first_gid + g;
    return play_lane<POS>(r0, gid, (u32)POS) | (play_lane<POS>(r1, gid + 1, (u32)POS) << 16);
}

// ---- lock-step path: every live game of the warp has made `hint` plays, so the trick position POS = hint & 3 is a
// compile-time constant: the mover is slot POS for everybody, the trick-position arithmetic and the trick-end branch fold.
// hm = slot POS (the mover's hand); POS < 3: n0 = slot POS + 1 (the next seat); POS == 3: n0, n1, n2 = slots 0, 1, 2.
template <bool RANDOM, int POS, bool MASK, bool BOTS = false>
__device__ __forceinline__ void step_game_lock(const Env& e, u32 g, u64& meta, u64& hm, u64& n0, u64& n1, u64& n2, u32 card,
                                               u32 x16, u64& next_mask, u32& log_out, const uint8_t* __restrict__ sel8, u64 fgid,
                                               u32 bm = 0u) {
    const u32 na = (u32)e.n_alloc;
    const u32 lo = (u32)meta, hi = (u32)(meta >> 32);
    const u32 leader = (lo >> M_LEADER) & 3u, kf = (lo >> M_KLOPFAM) & 1u;
    const u32 mover = (leader + (u32)POS) & 3u;
    const u32 plays = (hi >> (M_PLAYS - 32)) & 63u;
    if (RANDOM) {
        const u64 legal = legal_moves(hm, POS != 0, hi & 63u, kf);
        card = nth_set_bit_lut(legal, play_pick(x16, e.rng, fgid + g, plays, (u32)__popcll(legal)), sel8);
    }
    if (BOTS) {                                                    // no byte-select table in shared memory here
        if (bm > 15u) { meta = input_error(e, meta); next_mask = 0; return; }
        if ((bm >> mover) & 1u) {
            const u64 legal = legal_moves(hm, POS != 0, hi & 63u, kf);
            card = nth_set_bit(legal, play_pick(x16, e.rng, fgid + g, plays, (u32)__popcll(legal)));
        }
    }
    PlayResult pr;
    meta = play_card<!RANDOM, POS, false>(meta, hm, card, 0ull, 0ull, pr);
    next_mask = 0;
    if (!RANDOM && ((meta >> M_ERR) & 1ull)) {                     // the hand is untouched; the caller stores it back as is
        atomicAdd((unsigned long long*)&e.stats[S_ERR_EVENTS], 1ull);
        return;
    }
    if (e.hist) e.hist[(u64)plays * na + g] = (uint8_t)((mover << 6) | card);
    if (POS < 3) {
        if (MASK) next_mask = legal_moves(n0, true, (u32)(meta >> 32) & 63u, kf);
    } else {
        log_out = log_entry((u32)(meta >> 32) & 0xFFFFFFu, pr.winner, (u32)meta);
        rotate4(n0, n1, n2, hm, pr.winner_rel);                    // slots 0..3 re-seated from the winner
        // the winner opens the next trick: everything it holds (minus the Klop-family pagat rule), nothing once finished
        if (MASK) next_mask = (((u32)meta >> M_PHASE) & 3u) == PH_PLAY ? legal_moves(n0, false, 0u, kf) : 0ull;
    }
}

// The work of a lock-step launch on one lane's game pair once its state is in registers: m = meta, hm = slot POS (the
// mover's hand), n0 = slot POS + 1 (MASK or POS == 3), n1 / n2 = slots 1 / 2 (POS == 3), rc = the draw-cache entry.
template <bool RANDOM, int POS, bool MASK, bool BOTS = false>
__device__ __forceinline__ void step_lock_body(const Env& e, u32 g, int hint, u64 fgid, u32 tag, bool cached, ulonglong2 m,
                                               ulonglong2 hm, ulonglong2 n0, ulonglong2 n1, ulonglong2 n2, uint2 rc, u32 act,
                                               const uint8_t* __restrict__ sel8, u32 bm2 = 0u) {
    const u32 na = (u32)e.n_alloc;
    const bool a0 = (((u32)m.x >> M_PHASE) & 3u) == PH_PLAY && (RANDOM || (act & 0xFFu) != CARD_SKIP),
               a1 = (((u32)m.y >> M_PHASE) & 3u) == PH_PLAY && (RANDOM || (act >> 8) != CARD_SKIP);
    // plays sit in the top byte of the high word and the bits above them are clear for every live game
    const bool in_step = (!a0 || ((u32)(m.x >> 32) >> (M_PLAYS - 32)) == (u32)hint)
                      && (!a1 || ((u32)(m.y >> 32) >> (M_PLAYS - 32)) == (u32)hint);
    const bool lock = __all_sync(0xFFFFFFFFu, in_step);            // the hint is only a hint: each warp checks it
    if (!a0 && !a1) return;
    if (!lock) { step_pair_general_cold<RANDOM, POS, MASK, BOTS>(e, g, m, a0, a1, act, hm, n0, n1, n2, bm2); return; }
    u32 x0 = 0, x1 = 0;                            // the two games' 16-bit lanes of this play
    if (RANDOM) {
        if (POS > 0 && cached && rc.x == tag) {
            x0 = rc.y & 0xFFFFu; x1 = rc.y >> 16;
        } else if (POS > 0 && cached) {            // a miss (stale or never-written entry): rare, out of line
            const u32 x = pair_lanes_cold<POS>(e, g, (u32)hint >> 2, a1);
            x0 = x & 0xFFFFu; x1 = x >> 16;
        } else {
            // the trick index is the (uniform) hint -- a finished neighbour's own counter is stale and must not be used
            Words4 r0, r1;
            pair_blocks(e, g, (u32)hint >> 2, (u32)hint >> 2, a1, r0, r1);
            x0 = play_lane<POS>(r0, fgid + g, (u32)hint);
            x1 = play_lane<POS>(r1, fgid + g + 1, (u32)hint);
            if (POS == 0 && cached) {
                uint2* rcp = e.rcache + (g >> 1);
                rcp[0] = make_uint2(tag, play_lanes_of_pair(r0, 1));
                rcp[na >> 1] = make_uint2(tag, play_lanes_of_pair(r0, 2));
                if (e.rc_rows > 2u) rcp[na] = make_uint2(tag, play_lanes_of_pair(r0, 3));
            }
        }
    }
    if (BOTS) {                                    // Philox only for a pair with a bot to move; the draw cache is neither read nor written
        const bool b1 = a1 && bot_moves(m.y, bm2 >> 8);
        if ((a0 && bot_moves(m.x, bm2 & 0xFFu)) || b1) {
            Words4 r0, r1;
            pair_blocks(e, g, (u32)hint >> 2, (u32)hint >> 2, b1, r0, r1);
            x0 = play_lane<POS>(r0, fgid + g, (u32)hint);
            x1 = play_lane<POS>(r1, fgid + g + 1, (u32)hint);
        }
    }
    u64 k0 = 0, k1 = 0;
    u32 l0 = 0, l1 = 0;                            // trick-log entries (POS == 3); 0 = nothing to append
    if (a0) step_game_lock<RANDOM, POS, MASK, BOTS>(e, g, m.x, hm.x, n0.x, n1.x, n2.x, act & 0xFFu, x0, k0, l0, sel8, fgid, bm2 & 0xFFu);
    if (a1) step_game_lock<RANDOM, POS, MASK, BOTS>(e, g + 1, m.y, hm.y, n0.y, n1.y, n2.y, act >> 8, x1, k1, l1, sel8, fgid, bm2 >> 8);
    st2(e.hands + (POS * na + g), hm.x, hm.y);     // a game that did not move gets its slot back unchanged
    if (POS == 3) {
        st2(e.hands + g, n0.x, n0.y); st2(e.hands + (na + g), n1.x, n1.y); st2(e.hands + (2 * na + g), n2.x, n2.y);
        // append-only trick log (4 B per game, coalesced) instead of a scattered read-modify-write of the winner's pile;
        // the trick index is the uniform hint.  (A game that refused an illegal card gets a 0 entry nobody reads.)
        u32* row = e.tricklog + (u64)((u32)hint >> 2) * na + g;   // 12 rows of n_alloc <= 2^29 entries: 64-bit index
        if (a0 && a1) *reinterpret_cast<uint2*>(row) = make_uint2(l0, l1);
        else if (a0) row[0] = l0;
        else row[1] = l1;
    }
    st2(e.meta + g, m.x, m.y);
    // an in-kernel pick is always legal and only the trick-closing play can end a game: nothing to clear at positions 0-2
    if (MASK || !RANDOM || POS == 3) store_masks<RANDOM, MASK>(e, g, m, a0, a1, k0, k1);
}

template <bool RANDOM, int POS, bool MASK, bool BOTS = false>
__device__ __forceinline__ void step_lock(const Env& e, const uint8_t* __restrict__ action, int hint, const uint8_t* __restrict__ bots) {
    const u32 g = (blockIdx.x * CTA + threadIdx.x) * 2;
    const u32 na = (u32)e.n_alloc;                 // the grid covers n_alloc exactly: no partial warps
    __shared__ __align__(16) uint8_t sel8[RANDOM ? SELECT8_SMEM : 16];
    uint2 sel8_mine = {0u, 0u};                    // this thread's 8 bytes of the byte-select table (tarok_rules.cuh): independent of
    if (RANDOM) sel8_mine = select8_fetch();       // the previous launch, so the load is issued before the dependency wait
    // the run parameters: launch parameters, overwritten from the device record first thing in the GRAPH kernel variants
    const u64 fgid = (RANDOM || BOTS) ? e.first_gid : 0ull;
    const u32 tag = (RANDOM ? e.rc_epoch : 0u) | ((u32)hint >> 2);
    pdl_wait();                                    // the previous step's writes are visible from here on
    // every load is issued before the first use: one memory round trip per step
    ulonglong2 m = ld2(e.meta + g);
    ulonglong2 hm = ld2(e.hands + (POS * na + g));
    ulonglong2 n0 = {0, 0}, n1 = {0, 0}, n2 = {0, 0};
    if (MASK || POS == 3) n0 = ld2(e.hands + (((POS + 1) & 3) * na + g));     // the next seat's slot is only read for its mask
    if (POS == 3) { n1 = ld2(e.hands + (na + g)); n2 = ld2(e.hands + (2 * na + g)); }
    u32 act = 0, bm2 = 0;
    if (!RANDOM) act = load_actions(action, g, e.n);
    if (BOTS) bm2 = load_actions(bots, g, e.n);   // the seat masks of the pair: one more coalesced 2-byte load
    // draw cache: the pair's Philox block is computed by the position-0 launch of a trick, which leaves the lanes of
    // positions 1-3 behind ({tag, lanes}, 8 B per pair and position); the three launches that follow read 8 B instead of
    // running the ten rounds again.  The tag (epoch of first_gid | trick) makes a stale or never-written entry harmless:
    // the block is then computed here as before.  Lanes straddle two pairs when first_gid is odd: no cache then.
    constexpr u32 UPOS = POS > 0 ? (u32)POS : 0u;
    bool in_rows = RANDOM && e.rc_rows != 0u;      // a launch parameter: the entry is fetched whatever first_gid turns out to be
    if constexpr (POS > 0) in_rows = in_rows && UPOS <= e.rc_rows;
    const bool cached = in_rows && !((u32)fgid & 1u);
    uint2 rc = {0u, 0u};
    if (in_rows && POS > 0) rc = e.rcache[(UPOS > 0u ? UPOS - 1u : 0u) * (na >> 1) + (g >> 1)];
    // the table is stored behind the state loads in program order, so all of them are in flight together (A/B against a store
    // before pdl_wait, profiles/r02/step_ab_run7.txt: 8.03 vs 8.14 us at 1 M, 71.9 vs 72.5 at 8 M)
    if (RANDOM) {
        select8_store(sel8, sel8_mine);
        __syncthreads();
    }
    step_lock_body<RANDOM, POS, MASK, BOTS>(e, g, hint, fgid, tag, cached, m, hm, n0, n1, n2, rc, act, sel8, bm2);
}

// `hint` = the number of plays every live game has made so far (lock-step pipelines know it on the host); POS = hint & 3
// is compiled in (one kernel per trick position, each with its own register allocation); POS = -1: no hint.
// MASK = write the legal mask of the next seat to move (the stepwise API: every launch a caller can observe).  A CHAIN of
// in-kernel random steps (tarok_steps_random, the stepwise rollouts) launches its interior steps with MASK = false: no
// caller can see those masks, so the next seat's slot is neither read nor its legal set computed or stored -- 16 of the
// 48 bytes a step moves at trick positions 0-2 -- and only the chain's last launch produces the masks.
// BOTS (with RANDOM = false): the third action source, tarok_step_bots -- `bots` = the per-game seat masks.
template <bool RANDOM, int POS, bool MASK = true, bool GRAPH = false, bool BOTS = false>
__global__ void __launch_bounds__(CTA, RANDOM ? ((POS >= 0 && POS < 3) ? TK_STEP_BLOCKS_RANDOM_012
                                                   : POS == 3 ? TK_STEP_BLOCKS_RANDOM_3 : TK_STEP_BLOCKS_RANDOM)
                                           : BOTS ? TK_STEP_BLOCKS_BOTS : TK_STEP_BLOCKS_FORCED)
k_step(Env e, const uint8_t* __restrict__ action, int hint, const uint8_t* __restrict__ bots) {
    pdl_launch_dependents();
    if constexpr (GRAPH) load_run_params(e);       // written before the graph started: no need to wait for the previous kernel
    if constexpr (POS >= 0) {
        step_lock<RANDOM, POS, MASK, BOTS>(e, action, hint, bots);
    } else {
        const u32 g = (blockIdx.x * CTA + threadIdx.x) * 2;
        pdl_wait();
        const ulonglong2 m = ld2(e.meta + g), z = {0, 0};
        u32 act = 0, bm2 = 0;
        if (!RANDOM) act = load_actions(action, g, e.n);
        if (BOTS) bm2 = load_actions(bots, g, e.n);
        const bool a0 = (((u32)m.x >> M_PHASE) & 3u) == PH_PLAY && (RANDOM || (act & 0xFFu) != CARD_SKIP),
                   a1 = (((u32)m.y >> M_PHASE) & 3u) == PH_PLAY && (RANDOM || (act >> 8) != CARD_SKIP);
        if (a0 || a1) step_pair_general<RANDOM, -1, MASK, BOTS>(e, g, m, a0, a1, act, z, z, z, z, bm2);
    }
}

// Seat-indexed copy of the hand slots (for callers that want Roka by seat rather than by trick position).
__global__ void __launch_bounds__(CTA) k_hands_by_seat(Env e, u64* __restrict__ out) {
    const u64 g = (u64)blockIdx.x * CTA + threadIdx.x;
    const u64 na = e.n_alloc;
    if (g >= na) return;
    u64 a = e.hands[g], b = e.hands[na + g], c = e.hands[2 * na + g], d = e.hands[3 * na + g];
    slots_to_seats(a, b, c, d, leader_of(e.meta[g]));
    out[g] = a; out[na + g] = b; out[2 * na + g] = c; out[3 * na + g] = d;
}

// Standalone legal mask, recomputed from hands + meta (24 B/env-step algorithmic).
__global__ void __launch_bounds__(CTA) k_legal_mask(Env e, u64* __restrict__ out) {
    u64 g = ((u64)blockIdx.x * CTA + threadIdx.x) * 2;
    if (g >= e.n_alloc) return;
    const u64 na = e.n_alloc;
    ulonglong2 m = ld2(e.meta + g);
    ulonglong2 h0 = ld2(e.hands + g), h1 = ld2(e.hands + na + g), h2 = ld2(e.hands + 2 * na + g),
               h3 = ld2(e.hands + 3 * na + g);
    // the seat to move sits in slot `pos`
    u64 k0 = mask_for_mover(m.x, sel4(h0.x, h1.x, h2.x, h3.x, mget(m.x, M_POS, 2)));
    u64 k1 = mask_for_mover(m.y, sel4(h0.y, h1.y, h2.y, h3.y, mget(m.y, M_POS, 2)));
    if (g + 1 < e.n) st2(out + g, k0, k1);
    else if (g < e.n) out[g] = k0;
}

// ------------------------------------------------------------------------------------------------
// score: Roka.prestej + the three start() epilogues; accumulates the statistics vector.
// 56 B/deal algorithmic: R 4 piles 32 + talon 8 + meta 8, W int16[4] 8.
// ------------------------------------------------------------------------------------------------
// Piles are materialised here (MAT): pile[s] = what the exchange laid down (stored) | the tricks seat s won (trick log);
// in Klop the talon loses the cards that went into tricks 1..6.  Idempotent.
__device__ __forceinline__ void materialise(u64 meta, const uint2* log12, int which, u64 order,
                                            u64& p0, u64& p1, u64& p2, u64& p3, u64& talon) {
    const u32 tricks = mget(meta, M_TRICKS, 4);
    const bool klop = mget(meta, M_CONTRACT, 4) == C_KLOP;
#pragma unroll
    for (u32 k = 0; k < 12; k++) {
        if (k < tricks) {
            const u32 entry = which ? log12[k].y : log12[k].x;
            u64 tc;
            const u64 b = trick_bits(entry, k, klop, order, tc);
            const u32 w = entry >> 30;
            p0 |= w == 0 ? b : 0ull; p1 |= w == 1 ? b : 0ull; p2 |= w == 2 ? b : 0ull; p3 |= w == 3 ? b : 0ull;
            talon &= ~tc;
        }
    }
}

// Scores straight from the trick log: every entry carries its winner and the card points of its four cards, and
// Roka.prestej is order independent -- sum(points) - 2 * floor(n / 3) - [n % 3 != 0] over the n cards of a pile
// (Roka.py:55-98) -- so no bitboard is rebuilt: per trick one compare-and-add.
//   Navadna / Solo (Navadna_igra.py:80-113): the team's points = the declarer's discards (`dpts`, k cards) + the tricks won by
//     a seat of `ekipa`; the leftover talon joins them iff a lone declarer in a king game took the called king (Q7) -- bit 29
//     of the entry of the trick that held it.
//   Klop (Klop.py:36-45): per seat; the talon card of tricks 1..6 (popped from the END, Klop.py:67-71) goes to the winner.
//   Berac (Berac.py:33-44): the game stops on the declarer's first trick, so "the declarer took a trick" = "the last
//     trick's winner is the declarer".
__device__ __forceinline__ u64 score_from_log(u64 meta, const uint2* log12, int which, u32 dpts, u64 talon, u64 order) {
    const u32 lo = (u32)meta;
    const u32 contract = lo & 15u, decl = (lo >> M_DECL) & 3u, tricks = (lo >> M_TRICKS) & 15u;
    if (is_navadna(contract)) {
        const u32 team = (lo >> M_TEAM) & 15u, king = (lo >> M_KING) & 7u;
        const u32 valid = (1u << tricks) - 1u;            // entries past the tricks played are stale
        // Four tricks at a time, one per byte: the top byte of an entry is points (5 bits) | called-king flag | winner (2 bits).
        // "won by the declarer's team" = bit `winner` of the 4-bit team mask, picked per byte with two select stages on
        // byte-replicated team bits; everything else is byte-parallel adds (no byte can overflow: <= 3 x 20 points).
        const u32 ONES = 0x01010101u;
        const u32 t0 = (team & 1u) * ONES, t1 = ((team >> 1) & 1u) * ONES, t2 = ((team >> 2) & 1u) * ONES, t3 = (team >> 3) * ONES;
        u32 accp = 0, accw = 0, acck = 0;
#pragma unroll
        for (u32 j = 0; j < 3; j++) {
            const u32 e0 = which ? log12[4 * j].y : log12[4 * j].x, e1 = which ? log12[4 * j + 1].y : log12[4 * j + 1].x,
                      e2 = which ? log12[4 * j + 2].y : log12[4 * j + 2].x, e3 = which ? log12[4 * j + 3].y : log12[4 * j + 3].x;
            const u32 top = __byte_perm(__byte_perm(e0, e1, 0x0073), __byte_perm(e2, e3, 0x0073), 0x5410);
            const u32 w0 = (top >> 6) & ONES, w1 = (top >> 7) & ONES;
            const u32 lo2 = (t0 & ~w0) | (t1 & w0), hi2 = (t2 & ~w0) | (t3 & w0);
            const u32 vj = (((valid >> (4 * j)) & 15u) * 0x00204081u) & ONES;        // the four valid bits, one per byte
            const u32 mine = ((lo2 & ~w1) | (hi2 & w1)) & vj;                         // 0 / 1 per byte
            accp += top & (mine * 0x1Fu);
            accw += mine;
            acck |= (top >> 5) & mine;
        }
        const u32 pts_won = (accp * ONES) >> 24, won = (accw * ONES) >> 24, kings = acck != 0u ? 1u : 0u;
        u32 pts = dpts + pts_won;
        u32 n = 4u * won + (((lo >> M_GROUP) & 7u) != NO_GROUP ? talon_k(contract) : 0u);
        // leftover talon to a lone declarer of a king game who took the called king (Q7); a lone declarer is the whole team
        if (contract != C_SOLO_BREZ && __popc(team) == 1 && king != NO_KING && (kings & 1u)) {
            pts += card_points(talon); n += (u32)__popcll(talon);
        }
        return score_navadna_v(meta, prestej_pn((int)pts, (int)n));
    }
    if (is_berac(contract)) return score_berac(meta, ((lo >> M_WINNER) & 3u) == decl);
    if (contract != C_KLOP) return 0ull;
    u32 acc = 0;                                          // per seat one byte: card points (<= 106) of the pile
    u32 cnt = 0;                                          // per seat one byte: cards
#pragma unroll
    for (u32 k = 0; k < 12; k++) {
        if (k < tricks) {
            const u32 entry = which ? log12[k].y : log12[k].x;
            u32 p = (entry >> 24) & 31u, c = 4u;
            if (k < 6) { p += card_points1((u32)(order >> (6 * (5 - k))) & 63u); c = 5u; }
            const u32 sh = 8u * (entry >> 30);
            acc += p << sh; cnt += c << sh;
        }
    }
    const int a = prestej_pn((int)(acc & 255u), (int)(cnt & 255u)), b = prestej_pn((int)((acc >> 8) & 255u), (int)((cnt >> 8) & 255u)),
              c = prestej_pn((int)((acc >> 16) & 255u), (int)((cnt >> 16) & 255u)), d = prestej_pn((int)(acc >> 24), (int)(cnt >> 24));
    const bool any = a > 35 || b > 35 || c > 35 || d > 35;
    return pack_scores(any ? 0 : -a, any ? 0 : -b, any ? 0 : -c, any ? 0 : -d);
}

// MAT = also write the materialised piles / talon back (the exported fields then hold the full piles); without it only the
// scores and statistics are produced (pipelines that, like Tarok.paralel_start, only need the results): what is read is
// meta 8 + trick log 48 + talon 8 + discard points 1 (+ the talon order for Klop), 8 B of scores written.
template <bool MAT, bool GRAPH = false>
__global__ void __launch_bounds__(CTA) k_score(Env e, u64* __restrict__ out, u64 out_n) {
    if constexpr (GRAPH) load_run_params(e);
    u64 g = ((u64)blockIdx.x * CTA + threadIdx.x) * 2;
    const u64 na = e.n_alloc;
    u64 s0 = 0, s1 = 0;
    bool f0 = false, f1 = false, e0 = false, e1 = false;
    u32 c0 = 0, c1 = 0, pl0 = 0, pl1 = 0;
    if (g < na) {
        ulonglong2 m = ld2(e.meta + g);
        ulonglong2 t = ld2(e.talon + g);
        const u32 dp = *reinterpret_cast<const unsigned short*>(e.dpts + g);
        uint2 log12[12];                                  // all twelve entries are fetched up front (one memory phase);
#pragma unroll                                            // entries past the tricks played are stale and never looked at
        for (u32 k = 0; k < 12; k++) log12[k] = *reinterpret_cast<const uint2*>(e.tricklog + k * na + g);
        c0 = mget(m.x, M_CONTRACT, 4); c1 = mget(m.y, M_CONTRACT, 4);
        ulonglong2 o = {0, 0};
        if (MAT || c0 == C_KLOP || c1 == C_KLOP) o = ld2(e.torder + g);
        if (MAT) {
            ulonglong2 p0 = ld2(e.piles + g), p1 = ld2(e.piles + na + g), p2 = ld2(e.piles + 2 * na + g),
                       p3 = ld2(e.piles + 3 * na + g);
            ulonglong2 tt = t;
            materialise(m.x, log12, 0, o.x, p0.x, p1.x, p2.x, p3.x, tt.x);
            materialise(m.y, log12, 1, o.y, p0.y, p1.y, p2.y, p3.y, tt.y);
            *reinterpret_cast<ulonglong2*>(e.piles + g) = p0; *reinterpret_cast<ulonglong2*>(e.piles + na + g) = p1;
            *reinterpret_cast<ulonglong2*>(e.piles + 2 * na + g) = p2; *reinterpret_cast<ulonglong2*>(e.piles + 3 * na + g) = p3;
            *reinterpret_cast<ulonglong2*>(e.talon + g) = tt;
        }
        e0 = ((m.x >> M_ERR) & 1ull) && g < e.n;
        e1 = ((m.y >> M_ERR) & 1ull) && g + 1 < e.n;
        f0 = mget(m.x, M_PHASE, 2) == PH_DONE && !((m.x >> M_ERR) & 1ull) && g < e.n;
        f1 = mget(m.y, M_PHASE, 2) == PH_DONE && !((m.y >> M_ERR) & 1ull) && g + 1 < e.n;
        pl0 = g < e.n ? mget(m.x, M_PLAYS, 6) : 0u; pl1 = g + 1 < e.n ? mget(m.y, M_PLAYS, 6) : 0u;
        // the (pre-materialisation) talon is what the Navadna epilogue needs: no exchange ever follows the first card
        if (f0) s0 = score_from_log(m.x, log12, 0, dp & 0xFFu, t.x, o.x);
        if (f1) s1 = score_from_log(m.y, log12, 1, dp >> 8, t.y, o.y);
        if (g + 1 < out_n) st2(out + g, s0, s1);
        else if (g < out_n) out[g] = s0;
    }
    // two games per lane: folded per lane before the warp reductions
    const u64 fgid = e.first_gid;
    GameStat gs[2] = {{f0, e0, s0, c0, pl0, fgid + g}, {f1, e1, s1, c1, pl1, fgid + g + 1}};
    accumulate_stats<2>(e.stats, gs);
}

// ------------------------------------------------------------------------------------------------
// fused rollout: deal -> contract -> exchange -> up to 48 random plays -> score with the whole game in
// registers (one lane = one game).  Same device functions, same Philox draws, hence bit-identical to
// the stepwise pipeline.  Not HBM-bound: 8 B/deal written.
// ------------------------------------------------------------------------------------------------
struct FusedGame { u64 h0, h1, h2, h3, p0, p1, p2, p3, talon, order, meta; };   // h0..h3: hand SLOTS (leader-relative)

// One card play of the fused rollout at trick position J (compile-time: the loop over a trick is unrolled).  The hands are
// kept in leader-relative slots here too: the mover is register hJ, no select chain and no conditional write-back; the four
// registers are re-seated from the winner when the trick closes.
template <int J>
__device__ __forceinline__ void fused_play(FusedGame& f, const Words4& blk, const Rng& rng, u64 gid, u32 trick, bool klop,
                                           uint8_t* hist_row, u64 na, const uint8_t* __restrict__ sel8, u32* log_row = nullptr) {
    u64& hand = J == 0 ? f.h0 : J == 1 ? f.h1 : J == 2 ? f.h2 : f.h3;
    const u64 legal = legal_moves(hand, J != 0, (u32)(f.meta >> 32) & 63u, klop);
    const u32 n = (u32)__popcll(legal);
    const u32 card = nth_set_bit_lut(legal, play_draw<J>(blk, rng, gid, trick * 4 + J, n), sel8);
    if (hist_row) hist_row[(u64)J * na] = (uint8_t)((((((u32)f.meta >> M_LEADER) + (u32)J) & 3u) << 6) | card);
    PlayResult pr;
    f.meta = play_card<false, J>(f.meta, hand, card, f.talon, f.order, pr);
    if (J == 3) {
        if (log_row) *log_row = log_entry((u32)(f.meta >> 32) & 0xFFFFFFu, pr.winner, (u32)f.meta);
        const u64 b = pr.pile_bits;
        f.p0 |= pr.winner == 0 ? b : 0ull; f.p1 |= pr.winner == 1 ? b : 0ull;
        f.p2 |= pr.winner == 2 ? b : 0ull; f.p3 |= pr.winner == 3 ? b : 0ull;
        f.talon &= ~pr.talon_clear;
        rotate4(f.h0, f.h1, f.h2, f.h3, pr.winner_rel);
    }
}

enum : int { DEALS_PHILOX = 0, DEALS_PERM = 1, DEALS_RECORD = 2 };

template <int DEALS>
__global__ void __launch_bounds__(CTA) k_rollout_fused(Env e, u32 mode, const uint8_t* __restrict__ perm,
                                                       const uint8_t* __restrict__ fc, const uint8_t* __restrict__ fd,
                                                       const uint8_t* __restrict__ fk, u64* __restrict__ out, int write_state,
                                                       u64 g0) {
    extern __shared__ __align__(16) uint8_t shp[];
    __shared__ __align__(16) uint8_t sel8[SELECT8_SMEM];  // byte-select table of the uniform picks (tarok_rules.cuh)
    select8_to_shared(sel8);                              // made visible by the barrier below (DEALS_PERM) or the one that follows
    const u64 base = g0 + (u64)blockIdx.x * CTA;          // g0: first game of this launch (chunked host pipeline)
    u64 g = base + threadIdx.x;
    const u64 na = e.n_alloc;
    const u64 gid = e.first_gid + g;
    if (DEALS == DEALS_RECORD) {
        // the CTA's 256 records (5120 B, 16-byte aligned: the tile starts at a multiple of 4 records) go through shared memory
        // with coalesced 16-byte loads; a lane then reads its five words at a stride of 5 banks (conflict-free).  The staging
        // buffer is n_alloc x 54 bytes, so the last tile may read past the records: those lanes are not live.
        const uint4* src = reinterpret_cast<const uint4*>(perm + base * RECORD_BYTES);
        for (u32 v = threadIdx.x; v < CTA * RECORD_BYTES / 16; v += CTA) reinterpret_cast<uint4*>(shp)[v] = src[v];
    }
    if (DEALS == DEALS_PERM) {
        const u64 total = e.n * 54ull, off = base * 54ull;
        const bool vec_ok = (((uintptr_t)perm) & 15u) == 0;
        for (u32 v = threadIdx.x; v < CTA * 54 / 16; v += CTA) {
            u64 b = off + (u64)v * 16;
            if (vec_ok && b + 16 <= total) *reinterpret_cast<uint4*>(shp + v * 16) = *reinterpret_cast<const uint4*>(perm + b);
            else for (int k = 0; k < 16; k++) shp[v * 16 + k] = (b + k < total) ? perm[b + k] : 0xFF;
        }
    }
    __syncthreads();
    bool live = g < e.n, err = false;
    u64 meta = meta_pad(), packed = 0;
    u64 h0 = 0, h1 = 0, h2 = 0, h3 = 0, p0 = 0, p1 = 0, p2 = 0, p3 = 0, talon = 0, order = 0;
    if (live) {
        Dealt d;
        bool ok = true;
        DealRecord rec = {0u, 0u, NO_KING};
        if (DEALS == DEALS_PERM) d = deal_from_perm(shp + threadIdx.x * 54, ok);
        else if (DEALS == DEALS_RECORD) d = deal_from_record(reinterpret_cast<const u32*>(shp) + threadIdx.x * (RECORD_BYTES / 4), rec, ok);
        else d = deal_philox(e.rng, gid);
        h0 = d.h0; h1 = d.h1; h2 = d.h2; h3 = d.h3; talon = d.talon; order = d.order;
        meta = meta_fresh();
        const Words4 sb = setup_block(e.rng, gid);       // the device-side pre-play decisions (contract unless forced, exchange)
        if (!ok) meta = mset(meta, M_PHASE, 2, PH_DONE) | (1ull << M_ERR);
        else {
            u32 contract, declarer, king;
            if (DEALS == DEALS_RECORD) { contract = rec.contract; declarer = rec.declarer; king = rec.king; }
            else if (fc) resolve_contract<SRC_FORCED>(e.rng, gid, mode, fc, fd, fk, g, sb, contract, declarer, king);
            else resolve_contract<SRC_SYNTH>(e.rng, gid, mode, nullptr, nullptr, nullptr, g, sb, contract, declarer, king);
            meta = begin_contract(meta, contract, declarer, king, h0, h1, h2, h3);
        }
        if (write_state && e.hands0) {                   // hands as dealt (zacetna_roka), by seat: the replay kernels start from them
            e.hands0[g] = h0; e.hands0[na + g] = h1; e.hands0[2 * na + g] = h2; e.hands0[3 * na + g] = h3;
        }
        u64 dout = 0;
        if (mget(meta, M_PHASE, 2) == PH_EXCHANGE) {
            u32 decl = mget(meta, M_DECL, 2);
            u64 hand = sel4(h0, h1, h2, h3, decl), pile = 0;
            bool ok2 = exchange_game<true>(e.rng, gid, mode == 17u, sb, meta, hand, pile, talon, order, 0u, 0ull, dout, sel8);
            if (!ok2) meta = mset(meta, M_PHASE, 2, PH_DONE) | (1ull << M_ERR);
            else {
                h0 = decl == 0 ? hand : h0; h1 = decl == 1 ? hand : h1; h2 = decl == 2 ? hand : h2; h3 = decl == 3 ? hand : h3;
                p0 = decl == 0 ? pile : p0; p1 = decl == 1 ? pile : p1; p2 = decl == 2 ? pile : p2; p3 = decl == 3 ? pile : p3;
            }
        }
        if (write_state) {
            if (e.discard) e.discard[g] = dout;
            e.dpts[g] = (uint8_t)card_points(dout);
        }
        const u32 contract = mget(meta, M_CONTRACT, 4);
        const bool klop = klop_rules(contract);
        seats_to_slots(h0, h1, h2, h3, leader_of(meta));
        FusedGame fg{h0, h1, h2, h3, p0, p1, p2, p3, talon, order, meta};
        for (u32 trick = 0; trick < 12 && mget(fg.meta, M_PHASE, 2) == PH_PLAY; trick++) {
            Words4 blk = play_block(e.rng, gid, trick);                // 4 plays = half of one Philox block
            uint8_t* hrow = (e.hist && write_state) ? e.hist + (u64)(trick * 4) * na + g : nullptr;
            fused_play<0>(fg, blk, e.rng, gid, trick, klop, hrow, na, sel8);
            fused_play<1>(fg, blk, e.rng, gid, trick, klop, hrow, na, sel8);
            fused_play<2>(fg, blk, e.rng, gid, trick, klop, hrow, na, sel8);
            fused_play<3>(fg, blk, e.rng, gid, trick, klop, hrow, na, sel8, write_state ? e.tricklog + (u64)trick * na + g : nullptr);
        }
        h0 = fg.h0; h1 = fg.h1; h2 = fg.h2; h3 = fg.h3; p0 = fg.p0; p1 = fg.p1; p2 = fg.p2; p3 = fg.p3;
        talon = fg.talon; meta = fg.meta;
        err = (meta >> M_ERR) & 1ull;
        if (!err && mget(meta, M_PHASE, 2) == PH_DONE) packed = score_game(meta, p0, p1, p2, p3, talon);
        if (out) out[g] = packed;
    }
    if (write_state && g < na) {                         // h0..h3 are slots already (identity for a game that never started)
        e.hands[g] = h0; e.hands[na + g] = h1; e.hands[2 * na + g] = h2; e.hands[3 * na + g] = h3;
        e.piles[g] = p0; e.piles[na + g] = p1; e.piles[2 * na + g] = p2; e.piles[3 * na + g] = p3;
        e.talon[g] = talon; e.torder[g] = order; e.meta[g] = meta; e.mask[g] = 0;
    }
    GameStat gs[1] = {{live && !err && mget(meta, M_PHASE, 2) == PH_DONE, live && err, packed,
                       mget(meta, M_CONTRACT, 4), live ? mget(meta, M_PLAYS, 6) : 0u, gid}};
    accumulate_stats<1>(e.stats, gs);
}

}  // namespace tk
