// Observation expansion on the device: Nevronski_igralec.stanje_v_vektor_rek_navadna (Igralec.py:453-533).
//
// For the seat to move of every selected game the reference builds, per decision, a list of float arrays
// from the game history; here one WARP builds them straight from the compact state (history bytes, hands as
// dealt, discards, talon order, meta) and writes fp32 in the reference's layout.  Write-dominated:
// (T*216 + extras) * 4 bytes per acting game (SURVEY.md 8d).
//
// Reference behaviour reproduced (SURVEY.md A.4 / Q16):
//  * T = n + (8 - n % 8) with n = len(zgodovina) counting EVERY entry: the plays, the ("Talon", ...) entry of an
//    exchange and the (None, card) entries of Klop talon cards (the filter at Igralec.py:457 is always true).
//  * rows advance on player plays only: row i = i-th card play.  nasprotniki[i, opp, card] for opponents'
//    plays; roka_input[i, :] for own plays = the hand AS DEALT (pre-exchange, Igralec.py:264,465) minus the own
//    cards played before row i (discards and talon pick-ups never change it).
//  * opponent index = position among the other three players in seat order; self = 3 (Igralec.py:271-274).
//  * talon_input: Navadna/Solo [6,55] row j = j-th talon card one-hot, column 54 = "in the chosen group"
//    (only once the exchange is in the history; Solo_brez never has one); Klop [54] multi-hot of the talon cards
//    revealed so far; Berac none.  zalozil[54] = own discards, only for the seat that exchanged.
//
// Element types: the observation kernels are templates over the OUTPUT type O (float, __nv_bfloat16, __half) and the
// selection kernels over the INPUT type Q of the network outputs.  Every observation value is exactly 0 or 1, so all three
// hold it exactly; network outputs are widened to fp32 (exact) before any comparison, so a selection on bf16 / fp16
// outputs is the fp32 selection of the widened values.  qmax / next_Q_max and the replay targets stay fp32.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "tarok_kernels.cuh"

namespace tk {

enum : int { NET_KLOP = 0, NET_NAVADNA = 1, NET_SOLO = 2, NET_BERAC = 3 };     // Nevronski_igralec.Tipi_NN

__device__ __forceinline__ u32 net_type_of(u32 contract) {       // tip_igre_v_tip_izbire, Igralec.py:179-188
    return contract == C_KLOP ? NET_KLOP : is_king_game(contract) ? NET_NAVADNA : is_berac(contract) ? NET_BERAC : NET_SOLO;
}
__device__ __forceinline__ u32 history_len(u64 meta) {
    const u32 contract = mget(meta, M_CONTRACT, 4);
    u32 n = mget(meta, M_PLAYS, 6);
    if (mget(meta, M_GROUP, 3) != NO_GROUP) n += 1;                                   // the ("Talon", ...) entry
    if (contract == C_KLOP) n += min(mget(meta, M_TRICKS, 4), 6u);                    // (None, talon card) entries
    return n;
}
__device__ __forceinline__ u32 padded_rows(u32 n) { return n + (8u - (n & 7u)); }

// Per game: net type (0..3, 255 = not waiting for a card) and T, so the host can bucket like predict_igraj_karto.
__global__ void __launch_bounds__(CTA) k_obs_shape(Env e, uint8_t* __restrict__ type_out, uint8_t* __restrict__ rows_out) {
    const u64 g = (u64)blockIdx.x * CTA + threadIdx.x;
    if (g >= e.n) return;
    const u64 meta = e.meta[g];
    const bool live = mget(meta, M_PHASE, 2) == PH_PLAY;
    type_out[g] = live ? (uint8_t)net_type_of(mget(meta, M_CONTRACT, 4)) : (uint8_t)255;
    rows_out[g] = live ? (uint8_t)padded_rows(history_len(meta)) : (uint8_t)0;
}

// ------------------------------------------------------------------------------------------------
// Device-side bucket partition of the games waiting for a card -- what predict_igraj_karto does on the host with one
// queue per net type (Igralec.py:316-342) for each of the four players of Tarok.paralel_start (player of seat s in game
// i = (s + i) % 4, Tarok.py:34): key = (player, net type, T / 8 - 1), 4 x 4 x 7 = 112 buckets (+ key 127 = not waiting).
// A stable counting sort in three launches: per-CTA histograms, one column scan per key, scatter.  The host reads the
// 128 counts once per step (one small D2H) and then walks the non-empty ranges of `sel`.
// ------------------------------------------------------------------------------------------------
constexpr u32 BUCKETS = 128, BUCKET_DEAD = 127;

__device__ __forceinline__ u32 bucket_key(const Env& e, u64 g, u32 players) {
    if (g >= e.n) return BUCKET_DEAD;
    const u64 meta = e.meta[g];
    if (mget(meta, M_PHASE, 2) != PH_PLAY) return BUCKET_DEAD;
    const u32 player = players > 1 ? (mover_of(meta) + (u32)(e.first_gid + g)) & 3u : 0u;
    return player * 28u + net_type_of(mget(meta, M_CONTRACT, 4)) * 7u + (padded_rows(history_len(meta)) / 8u - 1u);
}

__global__ void __launch_bounds__(CTA) k_bucket_hist(Env e, u32 players, u32* __restrict__ cta_hist) {
    __shared__ u32 sh[BUCKETS];
    if (threadIdx.x < BUCKETS) sh[threadIdx.x] = 0;
    __syncthreads();
    const u32 key = bucket_key(e, (u64)blockIdx.x * CTA + threadIdx.x, players);
    // one shared atomic per distinct key per warp
    const u32 peers = __match_any_sync(0xFFFFFFFFu, key);
    if ((threadIdx.x & 31u) == (u32)__ffs(peers) - 1u) atomicAdd(&sh[key], (u32)__popc(peers));
    __syncthreads();
    if (threadIdx.x < BUCKETS) cta_hist[(u64)blockIdx.x * BUCKETS + threadIdx.x] = sh[threadIdx.x];
}

// One CTA of 128 x SCAN_PARTS threads: column k of cta_hist (one entry per CTA of the histogram kernel) becomes exclusive
// offsets in CTA order and its total counts[k] -- SCAN_PARTS threads per column, each over a contiguous range of CTAs (load
// all, local exclusive scan, add the sum of the ranges before it), instead of one thread walking the whole column; then an
// exclusive scan over the keys gives the bucket bases, counts[128 + k] (counts[255] = all listed games), and the bases in
// observation ROWS, counts[256 + k] = sum over earlier buckets of size * T (where a bucket's block of the [rows, 3, 54] /
// [rows, 54] arenas starts).
constexpr u32 SCAN_PARTS = 8;
__global__ void __launch_bounds__(BUCKETS * SCAN_PARTS) k_bucket_scan(u32* __restrict__ cta_hist, u32 n_cta, u32* __restrict__ counts) {
    __shared__ u32 part[SCAN_PARTS][BUCKETS];
    __shared__ u32 tot[BUCKETS];
    const u32 k = threadIdx.x % BUCKETS, p = threadIdx.x / BUCKETS;
    const u32 per = (n_cta + SCAN_PARTS - 1) / SCAN_PARTS, lo = p * per, hi = min(lo + per, n_cta);
    u32 sum = 0;
    for (u32 c = lo; c < hi; c++) sum += cta_hist[(u64)c * BUCKETS + k];
    part[p][k] = sum;
    __syncthreads();
    u32 run = 0;
    for (u32 q = 0; q < p; q++) run += part[q][k];
    for (u32 c = lo; c < hi; c++) {
        const u32 v = cta_hist[(u64)c * BUCKETS + k];
        cta_hist[(u64)c * BUCKETS + k] = run;
        run += v;
    }
    if (p == SCAN_PARTS - 1) tot[k] = k == BUCKET_DEAD ? 0u : run;      // games not waiting for a card are not listed
    __syncthreads();
    if (threadIdx.x == 0) {
        u32 base = 0, rows = 0;
        for (u32 j = 0; j < BUCKETS; j++) {
            const u32 v = tot[j];
            counts[j] = v; counts[BUCKETS + j] = base; counts[2 * BUCKETS + j] = rows;
            base += v; rows += v * 8u * (j % 7u + 1u);
        }
    }
}

__global__ void __launch_bounds__(CTA) k_bucket_scatter(Env e, u32 players, const u32* __restrict__ cta_hist,
                                                        const u32* __restrict__ counts, int* __restrict__ sel,
                                                        uint8_t* __restrict__ selkey) {
    __shared__ u32 warp_hist[CTA / 32][BUCKETS];
    for (u32 i = threadIdx.x; i < (CTA / 32) * BUCKETS; i += CTA) (&warp_hist[0][0])[i] = 0;
    __syncthreads();
    const u64 g = (u64)blockIdx.x * CTA + threadIdx.x;
    const u32 key = bucket_key(e, g, players);
    const u32 lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const u32 peers = __match_any_sync(0xFFFFFFFFu, key);
    const u32 rank = (u32)__popc(peers & ((1u << lane) - 1u));                  // stable: lower lanes first
    if (rank == 0) warp_hist[warp][key] = (u32)__popc(peers);
    __syncthreads();
    if (key == BUCKET_DEAD) return;
    u32 before = 0;
    for (u32 w = 0; w < warp; w++) before += warp_hist[w][key];
    const u32 at = counts[BUCKETS + key] + cta_hist[(u64)blockIdx.x * BUCKETS + key] + before + rank;
    sel[at] = (int)g;
    if (selkey) selkey[at] = (uint8_t)key;
}

template <class O> struct ObsOut {
    O* opp;          // [n_sel, T, 3, 54]
    O* hand;         // [n_sel, T, 54]
    O* talon;        // [n_sel, 6, 55] (Navadna, Solo) | [n_sel, 54] (Klop) | unused (Berac)
    O* king;         // [n_sel, 4]      (Navadna)
    O* decl;         // [n_sel, 4]      (Navadna, Solo, Berac)
    O* discard;      // [n_sel, 54]     (Navadna, Solo)
    O* mozne;        // [n_sel, 54]
    uint8_t* ok;     // [n_sel] 1 = game matched (net_type, T) and was expanded
};

// 0 or 1 as an observation element (b is 0 or 1): 1.0 is 0x3F80 in bf16 and 0x3C00 in fp16.
template <class O> __device__ __forceinline__ O obs_bit(u64 b);
template <> __device__ __forceinline__ float obs_bit<float>(u64 b) { return (float)b; }
template <> __device__ __forceinline__ __nv_bfloat16 obs_bit<__nv_bfloat16>(u64 b) { return __ushort_as_bfloat16((unsigned short)(b * 0x3F80u)); }
template <> __device__ __forceinline__ __half obs_bit<__half>(u64 b) { return __ushort_as_half((unsigned short)(b * 0x3C00u)); }

__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }

// Zero fill in element pairs: 8-byte stores for fp32, 4-byte stores for the half types.  count % 2 == 0, p aligned to a pair.
template <class O> __device__ __forceinline__ void warp_zero(O* p, u32 count, u32 lane) {
    if constexpr (sizeof(O) == 4) {
        float2* q = reinterpret_cast<float2*>(p);
        for (u32 i = lane; i < count / 2; i += 32) q[i] = make_float2(0.f, 0.f);
    } else {
        u32* q = reinterpret_cast<u32*>(p);
        for (u32 i = lane; i < count / 2; i += 32) q[i] = 0u;
    }
}
// Zero fill in 16-byte stores: count * sizeof(O) % 16 == 0, p 16-byte aligned.
template <class O> __device__ __forceinline__ void warp_zero4(O* p, u32 count, u32 lane) {
    if constexpr (sizeof(O) == 4) {
        float4* q = reinterpret_cast<float4*>(p);
        for (u32 i = lane; i < count / 4; i += 32) q[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    } else {
        uint4* q = reinterpret_cast<uint4*>(p);
        for (u32 i = lane; i < count / 8; i += 32) q[i] = make_uint4(0u, 0u, 0u, 0u);
    }
}
template <class O> __device__ __forceinline__ void warp_bits(O* p, u64 bits, u32 lane) {     // 54 elements from a bitboard
    p[lane] = obs_bit<O>((bits >> lane) & 1ull);
    if (lane + 32 < 54) p[lane + 32] = obs_bit<O>((bits >> (lane + 32)) & 1ull);
}

// `upto` < 0: the observation of the seat to move NOW.  `upto` = t >= 0: the observation the seat that made play t
// had at that decision (history truncated to the first t plays) -- the `stanje` of a replay sample; the legal-mask
// vector is not produced in that mode (it is not a network input, Igralec.py:333).
// One warp expands one game; `o` points at THIS game's blocks (null = not wanted).  Half outputs: opp / hand (T * 324 and
// T * 108 bytes, 16-byte multiples as T % 8 == 0) are zeroed in 16-byte stores, talon / discard / mozne / king / decl in
// 4-byte stores (their blocks are even element counts at 4-byte aligned starts).
template <class O>
__device__ __forceinline__ void obs_expand_game(const Env& e, u64 g, int net_type, u32 T, const ObsOut<O>& o, int upto, u32 lane) {
    const u64 na = e.n_alloc;
    const bool in_range = g < e.n;
    u64 meta = in_range ? e.meta[g] : meta_pad();
    const u32 contract = mget(meta, M_CONTRACT, 4);
    u32 self_at = 0;
    if (upto >= 0) {                                     // rewind the counters of meta to "before play upto"
        const bool had = (u32)upto < mget(meta, M_PLAYS, 6) && !((meta >> M_ERR) & 1ull);
        self_at = had ? (u32)(e.hist[(u64)upto * na + g] >> 6) : 0u;
        meta = mset(meta, M_PLAYS, 6, (u32)upto);
        meta = mset(meta, M_TRICKS, 4, (u32)upto >> 2);
        meta = mset(meta, M_PHASE, 2, had ? (u32)PH_PLAY : (u32)PH_DONE);
    }
    const u32 plays = mget(meta, M_PLAYS, 6);
    const bool match = mget(meta, M_PHASE, 2) == PH_PLAY && net_type_of(contract) == (u32)net_type
                    && padded_rows(history_len(meta)) == T;
    O* opp = o.opp;
    O* hand = o.hand;
    warp_zero4(opp, T * 162u, lane);                                 // T % 8 == 0: both blocks are 16-byte multiples
    warp_zero4(hand, T * 54u, lane);
    if (o.talon && net_type != NET_BERAC) warp_zero(o.talon, net_type == NET_KLOP ? 54u : 330u, lane);
    if constexpr (sizeof(O) == 4) {
        if (o.king && lane < 4) o.king[lane] = 0.f;
        if (o.decl && lane < 4) o.decl[lane] = 0.f;
    } else {
        if (o.king) warp_zero(o.king, 4u, lane);
        if (o.decl) warp_zero(o.decl, 4u, lane);
    }
    if (o.discard) warp_zero(o.discard, 54u, lane);
    if (o.mozne) warp_zero(o.mozne, 54u, lane);
    if (o.ok && lane == 0) *o.ok = match ? 1 : 0;
    __syncwarp();                                                    // zero fill ordered before the ones below
    if (!match) return;

    const u32 self = upto >= 0 ? self_at : mover_of(meta);
    const u32 decl = mget(meta, M_DECL, 2);
    // the two history slots of this lane: plays lane and lane + 32
    u32 h0 = 0xFF, h1 = 0xFF;
    if (lane < plays) h0 = e.hist[(u64)lane * na + g];
    if (lane + 32 < plays) h1 = e.hist[(u64)(lane + 32) * na + g];
    const bool own0 = h0 != 0xFF && (h0 >> 6) == self, own1 = h1 != 0xFF && (h1 >> 6) == self;
    // opponents' plays: one 1.0 each
    if (h0 != 0xFF && !own0) { u32 s = h0 >> 6; opp[(u64)lane * 162u + (s < self ? s : s - 1) * 54u + (h0 & 63u)] = obs_bit<O>(1); }
    if (h1 != 0xFF && !own1) { u32 s = h1 >> 6; opp[(u64)(lane + 32) * 162u + (s < self ? s : s - 1) * 54u + (h1 & 63u)] = obs_bit<O>(1); }
    // own plays: exclusive prefix-OR of the own cards played before each row (warp scan over 64 slots)
    u64 b0 = own0 ? 1ull << (h0 & 63u) : 0ull, b1 = own1 ? 1ull << (h1 & 63u) : 0ull;
    u64 inc0 = b0, inc1 = b1;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        u64 t0 = __shfl_up_sync(0xFFFFFFFFu, inc0, d), t1 = __shfl_up_sync(0xFFFFFFFFu, inc1, d);
        if (lane >= (u32)d) { inc0 |= t0; inc1 |= t1; }
    }
    const u64 all0 = __shfl_sync(0xFFFFFFFFu, inc0, 31);
    const u64 before0 = inc0 & ~b0, before1 = (all0 | inc1) & ~b1;   // own cards are distinct, so "& ~own" = exclusive
    const u64 dealt = e.hands0[self * na + g];
    u32 rows0 = __ballot_sync(0xFFFFFFFFu, own0), rows1 = __ballot_sync(0xFFFFFFFFu, own1);
    while (rows0) {
        const u32 src = __ffs(rows0) - 1; rows0 &= rows0 - 1;
        warp_bits(hand + (u64)src * 54u, dealt & ~__shfl_sync(0xFFFFFFFFu, before0, src), lane);
    }
    while (rows1) {
        const u32 src = __ffs(rows1) - 1; rows1 &= rows1 - 1;
        warp_bits(hand + (u64)(src + 32) * 54u, dealt & ~__shfl_sync(0xFFFFFFFFu, before1, src), lane);
    }
    // small vectors
    const u64 order = e.torder[g];
    if (o.talon && net_type == NET_KLOP) {
        const u32 shown = min(mget(meta, M_TRICKS, 4), 6u);           // Klop.py:69 pops from the end
        if (lane < shown) o.talon[(order >> (6 * (5 - lane))) & 63ull] = obs_bit<O>(1);
    } else if (o.talon && (net_type == NET_NAVADNA || net_type == NET_SOLO)) {
        const u32 grp = mget(meta, M_GROUP, 3), k = talon_k(contract);
        if (grp != NO_GROUP && lane < 6) {
            O* row = o.talon + lane * 55u;
            row[(order >> (6 * lane)) & 63ull] = obs_bit<O>(1);
            if (lane / k == grp) row[54] = obs_bit<O>(1);
        }
    }
    if (o.king && lane == 0) { u32 kg = mget(meta, M_KING, 3); if (kg < 4) o.king[kg] = obs_bit<O>(1); }
    if (o.decl && lane == 0) o.decl[decl == self ? 3u : (decl < self ? decl : decl - 1)] = obs_bit<O>(1);
    if (o.discard && self == decl && mget(meta, M_GROUP, 3) != NO_GROUP) warp_bits(o.discard, e.discard[g], lane);
    if (o.mozne && upto < 0) warp_bits(o.mozne, e.mask[g], lane);
}

// One (net type, T) bucket: `o` holds the bases of the bucket's arrays, game i of the selection gets block i.
template <class O>
__global__ void __launch_bounds__(CTA) k_obs_expand(Env e, int net_type, u32 T, const int* __restrict__ sel, u64 n_sel,
                                                    ObsOut<O> o, int upto) {
    const u32 lane = threadIdx.x & 31u;
    const u64 i = ((u64)blockIdx.x * CTA + threadIdx.x) >> 5;        // one warp per selected game
    if (i >= n_sel) return;
    const u64 g = sel ? (u64)sel[i] : i;
    ObsOut<O> m;
    m.opp = o.opp + i * (u64)T * 162u;
    m.hand = o.hand + i * (u64)T * 54u;
    m.talon = o.talon ? o.talon + i * (net_type == NET_KLOP ? 54u : 330u) : nullptr;
    m.king = o.king ? o.king + i * 4u : nullptr;
    m.decl = o.decl ? o.decl + i * 4u : nullptr;
    m.discard = o.discard ? o.discard + i * 54u : nullptr;
    m.mozne = o.mozne ? o.mozne + i * 54u : nullptr;
    m.ok = o.ok ? o.ok + i : nullptr;
    obs_expand_game(e, g, net_type, T, m, upto, lane);
}

// EVERY bucket of a step in one launch (after tarok_obs_buckets): position i of `sel` belongs to bucket selkey[i] =
// player * 28 + net * 7 + (T / 8 - 1); its rows go to the bucket's block of the arenas -- opp / hand at row counts[256 + key]
// + (i - counts[128 + key]) * T, the per-game vectors at index i -- so that each bucket's inputs are contiguous tensors.
template <class O> struct ObsArena { O* opp; O* hand; O* talon; O* talon_klop; O* king; O* decl; O* discard; };

template <class O>
__global__ void __launch_bounds__(CTA) k_obs_expand_all(Env e, const int* __restrict__ sel, const uint8_t* __restrict__ selkey,
                                                        const u32* __restrict__ counts, u64 n_total, ObsArena<O> a) {
    const u32 lane = threadIdx.x & 31u;
    const u64 i = ((u64)blockIdx.x * CTA + threadIdx.x) >> 5;
    if (i >= n_total) return;
    const u32 key = selkey[i];
    const u32 net = (key % 28u) / 7u, T = 8u * (key % 7u + 1u);
    const u64 row = (u64)counts[2 * BUCKETS + key] + (i - counts[BUCKETS + key]) * T;
    ObsOut<O> m;
    m.opp = a.opp + row * 162u;
    m.hand = a.hand + row * 54u;
    m.talon = net == NET_KLOP ? a.talon_klop + i * 54u : net == NET_BERAC ? nullptr : a.talon + i * 330u;
    m.king = net == NET_NAVADNA ? a.king + i * 4u : nullptr;
    m.decl = net != NET_KLOP ? a.decl + i * 4u : nullptr;
    m.discard = (net == NET_NAVADNA || net == NET_SOLO) ? a.discard + i * 54u : nullptr;
    m.mozne = nullptr;
    m.ok = nullptr;
    obs_expand_game(e, (u64)sel[i], (int)net, T, m, -1, lane);
}

// ------------------------------------------------------------------------------------------------
// Action selection on the device: Nevronski_igralec.igraj_karto (Igralec.py:344-355).
//   id = argmax(p[mozne_id]); karta = mozne[id]; next_Q_max = p[karta]; with probability random_card a uniform
//   legal card instead.  np.argmax returns the FIRST maximum in the order of the list `mozne`, so ties are broken
//   by that order (A.2): when following suit / trumping it is the player's suit list -- the cards as dealt in
//   ascending order, then the cards picked up from the talon in talon order (Roka.py:10-11,19-21); otherwise all
//   cards sorted ascending.  np.argmax also returns the first NaN, and a legal card is chosen whatever its value
//   (-inf, -FLT_MAX), so a diverged network still plays legal cards.  One warp per game; lanes hold cards lane and lane+32.
// ------------------------------------------------------------------------------------------------
enum : u32 { ST_EXPLORE = 8 };

// The order np.argmax ranks values by: NaN above everything (the first NaN wins), then the usual order, so that -inf and
// -FLT_MAX are ordinary values that any legal card can hold.  `a` ranks strictly above `b`:
__device__ __forceinline__ bool ranks_above(float a, float b) { return a > b || (a != a && b == b); }

// random.random() < random_card with random.random() = w / 2^32: `explore_threshold` = random_card * 2^32 (0 = never,
// 2^32 = always), so random_card = 1 explores at every word, 0xFFFFFFFF included.
__device__ __forceinline__ bool explores(u32 w, u64 explore_threshold) { return (u64)w < explore_threshold; }

template <class Q>
__device__ __forceinline__ void select_game(const Env& e, u64 g, const Q* __restrict__ qrow, u64 explore_threshold,
                                            uint8_t* __restrict__ card_out, float* __restrict__ qmax_out, u32 lane) {
    const u64 na = e.n_alloc;
    const u64 meta = e.meta[g];
    if (mget(meta, M_PHASE, 2) != PH_PLAY) { if (lane == 0) card_out[g] = 0xFF; return; }
    const u64 legal = e.mask[g];
    const u32 self = mover_of(meta);
    const u32 pos = mget(meta, M_POS, 2), lead = mget(meta, M_TRICK, 6);
    const u64 hand = e.hands[pos * na + g];                        // hand slots are leader-relative: the mover sits in slot pos
    // is `mozne` one of the player's own suit lists (list order) or the sorted union (id order)?
    bool list_order = false;
    if (pos != 0) list_order = (hand & suit_mask_of(lead)) != 0 || (hand & TAROKS) != 0;
    // the cards the declarer picked up from the talon (they follow the dealt cards in its suit lists, in talon order)
    const u64 order = e.torder[g];
    const u32 grp = mget(meta, M_GROUP, 3);
    const u64 picked = grp != NO_GROUP && self == mget(meta, M_DECL, 2)
                     ? talon_group_bits(order, talon_k(mget(meta, M_CONTRACT, 4)), grp) : 0ull;
    // "no card yet" = (-inf, key above every real key): any legal card beats it, whatever its value
    float best = -INFINITY;
    u32 best_key = 0xFFFFFFFFu, best_card = 0xFF;
#pragma unroll
    for (int h = 0; h < 2; h++) {
        const u32 c = lane + 32u * h;
        if (c < 54 && ((legal >> c) & 1ull)) {
            u32 key = c;
            if (list_order && ((picked >> c) & 1ull)) {          // picked up from the talon: after the dealt cards
                u32 tp = 0;
                for (u32 j = 0; j < 6; j++) if (((order >> (6 * j)) & 63ull) == c) tp = j;
                key = 64u + tp;
            }
            const float v = to_f32(qrow[c]);
            if (ranks_above(v, best) || (!ranks_above(best, v) && key < best_key)) { best = v; best_key = key; best_card = c; }
        }
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        const float ov = __shfl_xor_sync(0xFFFFFFFFu, best, d);
        const u32 ok = __shfl_xor_sync(0xFFFFFFFFu, best_key, d), oc = __shfl_xor_sync(0xFFFFFFFFu, best_card, d);
        if (ranks_above(ov, best) || (!ranks_above(best, ov) && ok < best_key)) { best = ov; best_key = ok; best_card = oc; }
    }
    if (lane == 0) {
        u32 card = best_card;
        if (explore_threshold) {                                  // random.random() < random_card (Igralec.py:352-353)
            const u64 gid = e.first_gid + g;
            const u32 plays = mget(meta, M_PLAYS, 6);
            Words4 b = philox_block(e.rng, gid, ST_EXPLORE, plays);
            if (explores(b.w[0], explore_threshold)) card = nth_set_bit(legal, draw_from_word(b.w[1], e.rng, gid, ST_EXPLORE, plays * 4 + 1, (u32)__popcll(legal)));
        }
        card_out[g] = (uint8_t)card;
        if (qmax_out) qmax_out[g] = best;                         // next_Q_max = p[argmax card] (Igralec.py:351)
        if (e.qmax_hist) e.qmax_hist[(u64)mget(meta, M_PLAYS, 6) * na + g] = best;   // kept for the replay targets
    }
}

template <class Q>
__global__ void __launch_bounds__(CTA) k_select_action(Env e, const Q* __restrict__ q, const int* __restrict__ sel,
                                                       u64 n_sel, u64 explore_threshold, uint8_t* __restrict__ card_out,
                                                       float* __restrict__ qmax_out) {
    const u32 lane = threadIdx.x & 31u;
    const u64 i = ((u64)blockIdx.x * CTA + threadIdx.x) >> 5;
    if (i >= n_sel) return;
    const u64 g = sel ? (u64)sel[i] : i;
    if (g >= e.n) return;
    select_game(e, g, q + i * 54u, explore_threshold, card_out, qmax_out, lane);
}

// The action selection of EVERY bucket of a step in one launch: qptr[key] = the [bucket size, 54] output of that bucket's
// forward pass (a table of device pointers the host fills), thr4[player] = the player's epsilon as a 32-bit threshold.
struct Thresholds4 { u64 t[4]; };
// The same with the table of bucket outputs passed BY VALUE (1 KB of kernel parameters): no device table to fill and copy.
// One element type for the whole table.
template <class Q> struct QTable { const Q* p[BUCKETS]; };
template <class Q>
__global__ void __launch_bounds__(CTA) k_select_action_all_tab(Env e, QTable<Q> qt, const int* __restrict__ sel,
                                                               const uint8_t* __restrict__ selkey, const u32* __restrict__ counts,
                                                               u64 n_total, Thresholds4 thr4, uint8_t* __restrict__ card_out,
                                                               float* __restrict__ qmax_out) {
    const u32 lane = threadIdx.x & 31u;
    const u64 i = ((u64)blockIdx.x * CTA + threadIdx.x) >> 5;
    if (i >= n_total) return;
    const u32 key = selkey[i];
    const Q* q = qt.p[key & (BUCKETS - 1)];
    if (!q) return;                                               // no forward was supplied for this bucket
    const u32 p = key / 28u;
    const u64 thr = p == 0 ? thr4.t[0] : p == 1 ? thr4.t[1] : p == 2 ? thr4.t[2] : thr4.t[3];
    select_game(e, (u64)sel[i], q + (i - counts[BUCKETS + key]) * 54u, thr, card_out, qmax_out, lane);
}

__global__ void __launch_bounds__(CTA) k_select_action_all(Env e, const float* const* __restrict__ qptr,
                                                           const int* __restrict__ sel, const uint8_t* __restrict__ selkey,
                                                           const u32* __restrict__ counts, u64 n_total, Thresholds4 thr4,
                                                           uint8_t* __restrict__ card_out, float* __restrict__ qmax_out) {
    const u32 lane = threadIdx.x & 31u;
    const u64 i = ((u64)blockIdx.x * CTA + threadIdx.x) >> 5;
    if (i >= n_total) return;
    const u32 key = selkey[i];
    const float* q = qptr[key];
    if (!q) return;                                               // no forward was supplied for this bucket
    const u32 p = key / 28u;
    const u64 thr = p == 0 ? thr4.t[0] : p == 1 ? thr4.t[1] : p == 2 ? thr4.t[2] : thr4.t[3];
    select_game(e, (u64)sel[i], q + (i - counts[BUCKETS + key]) * 54u, thr, card_out, qmax_out, lane);
}

// ------------------------------------------------------------------------------------------------
// Bidding and talon-exchange side of the neural player.
//   hand observation (pripavi_licitiram, Igralec.py:278-281): 54 multi-hot of each seat's hand;
//   exchange observation (menjaj_talon_v_vektor, Igralec.py:535-543): [hand 54, talon (54,6) card x group,
//     game one-hot 15 (igra_zalozi2index: (Tri|Dve|Ena, suit) -> 0..11, Solo_tri/dve/ena -> 12..14)];
//   exchange decision (menjaj_iz_talona, Igralec.py:365-385): group = first argmax of p[54:54+groups]; discards =
//     the st_kart best-valued cards of mozno_zalozit() after the pick-up, np.argsort()[-k:].  Among EQUAL values
//     numpy's order is build-dependent (its SIMD sorts are not stable), so ties are unpinned; here they go to the later
//     card in the order of mozno_zalozit (suits in Barva order, inside a suit the hand ascending, then the picked-up
//     cards in talon order), i.e. what a stable sort gives.  Each of the two choices is replaced by a uniform one
//     with probability random_card.
// ------------------------------------------------------------------------------------------------
template <class O>
__global__ void __launch_bounds__(CTA) k_obs_hands(Env e, O* __restrict__ out) {
    const u32 lane = threadIdx.x & 31u;
    const u64 g = ((u64)blockIdx.x * CTA + threadIdx.x) >> 5;
    if (g >= e.n) return;
    const u64 na = e.n_alloc;
    const u32 leader = leader_of(e.meta[g]);
#pragma unroll
    for (int s = 0; s < 4; s++) warp_bits(out + (g * 4 + s) * 54u, e.hands[slot_of((u32)s, leader) * na + g], lane);
}

// Half outputs: hand [54] and talon [324] in 4-byte stores, the game one-hot [15] (30 bytes, so game i starts 2-byte aligned
// only) in 2-byte stores.
template <class O>
__global__ void __launch_bounds__(CTA) k_obs_exchange(Env e, const int* __restrict__ sel, u64 n_sel, O* __restrict__ hand,
                                                      O* __restrict__ talon, O* __restrict__ game, uint8_t* __restrict__ ok) {
    const u32 lane = threadIdx.x & 31u;
    const u64 i = ((u64)blockIdx.x * CTA + threadIdx.x) >> 5;
    if (i >= n_sel) return;
    const u64 g = sel ? (u64)sel[i] : i;
    const u64 na = e.n_alloc;
    const u64 meta = g < e.n ? e.meta[g] : meta_pad();
    const bool match = mget(meta, M_PHASE, 2) == PH_EXCHANGE;
    warp_zero(hand + i * 54u, 54u, lane);
    warp_zero(talon + i * 324u, 324u, lane);
    if (lane < 15) game[i * 15u + lane] = obs_bit<O>(0);
    if (ok && lane == 0) ok[i] = match ? 1 : 0;
    __syncwarp();
    if (!match) return;
    const u32 contract = mget(meta, M_CONTRACT, 4), decl = mget(meta, M_DECL, 2), king = mget(meta, M_KING, 3);
    const u32 k = talon_k(contract);
    warp_bits(hand + i * 54u, e.hands[slot_of(decl, leader_of(meta)) * na + g], lane);
    const u64 order = e.torder[g];
    if (lane < 6) talon[i * 324u + ((order >> (6 * lane)) & 63ull) * 6u + lane / k] = obs_bit<O>(1);
    if (lane == 0) game[i * 15u + (is_king_game(contract) ? (contract - C_TRI) * 4u + king : 12u + (contract - C_SOLO_TRI))] = obs_bit<O>(1);
}

template <class Q>
__global__ void __launch_bounds__(CTA) k_select_exchange(Env e, const Q* __restrict__ p, const int* __restrict__ sel, u64 n_sel,
                                                         u64 explore_threshold, uint8_t* __restrict__ group_out,
                                                         u64* __restrict__ discard_out) {
    const u32 lane = threadIdx.x & 31u;
    const u64 i = ((u64)blockIdx.x * CTA + threadIdx.x) >> 5;
    if (i >= n_sel) return;
    const u64 g = sel ? (u64)sel[i] : i;
    if (g >= e.n) return;
    const u64 na = e.n_alloc;
    const u64 meta = e.meta[g];
    if (mget(meta, M_PHASE, 2) != PH_EXCHANGE) { if (lane == 0) { group_out[g] = 0xFF; discard_out[g] = 0; } return; }
    const u32 contract = mget(meta, M_CONTRACT, 4), decl = mget(meta, M_DECL, 2);
    const u32 k = talon_k(contract), groups = 6u / k;
    const u64 gid = e.first_gid + g;
    const unsigned full = 0xFFFFFFFFu;
    // group: first argmax of p[54 .. 54+groups)
    // (NaN first, the first maximum); the inactive lanes hold (-inf, 0xFF), which every real group beats
    float bv = lane < groups ? to_f32(p[i * 60u + 54u + lane]) : -INFINITY;
    u32 bi = lane < groups ? lane : 0xFFu;
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        const float ov = __shfl_xor_sync(full, bv, d);
        const u32 oi = __shfl_xor_sync(full, bi, d);
        if (ranks_above(ov, bv) || (!ranks_above(bv, ov) && oi < bi)) { bv = ov; bi = oi; }
    }
    u32 group = bi;
    Words4 rnd = philox_block(e.rng, gid, ST_EXPLORE, 50u);                       // same words on every lane
    if (explore_threshold && explores(rnd.w[0], explore_threshold)) group = draw_from_word(rnd.w[1], e.rng, gid, ST_EXPLORE, 201u, groups);
    const u64 order = e.torder[g];
    const u64 hand = e.hands[slot_of(decl, leader_of(meta)) * na + g];
    const u64 gb = talon_group_bits(order, k, group);
    u64 avail = (hand | gb) & DISCARDABLE;
    u64 discard = 0;
    if ((u32)__popcll(avail) < k) { if (lane == 0) { group_out[g] = (uint8_t)group; discard_out[g] = 0; } return; }   // Q19
    if (explore_threshold && explores(rnd.w[2], explore_threshold)) {              // random.sample(mozno, st_kart)
        Words4 r2 = philox_block(e.rng, gid, ST_EXPLORE, 51u);
        for (u32 j = 0; j < k; j++) {
            const u32 w = j == 0 ? r2.w[0] : j == 1 ? r2.w[1] : r2.w[2];
            const u64 bit = 1ull << nth_set_bit(avail, draw_from_word(w, e.rng, gid, ST_EXPLORE, 204u + j, (u32)__popcll(avail)));
            avail ^= bit; discard |= bit;
        }
    } else {
        for (u32 j = 0; j < k; j++) {                                              // k times: warp arg-max by (value, position)
            // NaN ranks highest (np.argsort sorts it last); key 0 = no card, below every real key
            float v = -INFINITY; u32 key = 0, card = 0xFF;
#pragma unroll
            for (int hh = 0; hh < 2; hh++) {
                const u32 c = lane + 32u * hh;
                if (c < 54 && ((avail >> c) & 1ull)) {
                    u32 pos = c & 63u;                                             // hand cards: ascending inside the suit
                    if (!((hand >> c) & 1ull)) {                                   // picked up: appended in talon order
                        u32 tp = 0;
                        for (u32 t = 0; t < 6; t++) if (((order >> (6 * t)) & 63ull) == c) tp = t;
                        pos = 64u + tp;
                    }
                    const u32 kk = (((c >= 32 ? 4u : (c >> 3)) << 8) | pos) + 1u;
                    const float pv = to_f32(p[i * 60u + c]);
                    if (ranks_above(pv, v) || (!ranks_above(v, pv) && kk > key)) { v = pv; key = kk; card = c; }
                }
            }
#pragma unroll
            for (int d = 16; d >= 1; d >>= 1) {
                const float ov = __shfl_xor_sync(full, v, d);
                const u32 ok2 = __shfl_xor_sync(full, key, d), oc = __shfl_xor_sync(full, card, d);
                if (ranks_above(ov, v) || (!ranks_above(v, ov) && ok2 > key)) { v = ov; key = ok2; card = oc; }
            }
            const u64 bit = 1ull << card;
            avail ^= bit; discard |= bit;
        }
    }
    if (lane == 0) { group_out[g] = (uint8_t)group; discard_out[g] = discard; }
}

// ------------------------------------------------------------------------------------------------
// Replay targets on the device: Nevronski_igralec.rezultat_stiha / rezultat_igre (Igralec.py:387-446).
// For every card play t of a finished game the reference stores a sample (stanje, dy) for the seat that played:
//   dy[c] = -70 for every card that was illegal at that decision (Igralec.py:393);
//   dy[card] = +vrednost_stiha(trick) if the seat took the trick else -vrednost_stiha(trick)  -- the Klop/Berac
//     branches compare a dict with a string and are dead (Q18); the 4- or 5-card trick counts sum-2 (Roka.py:92-95);
//   dy[card] += final_reword_factor * next, next = the seat's next_Q_max at its decision in the FOLLOWING trick, or for
//     its last sample the final score (st_tock; for Berac non-declarers -20 if all 12 tricks were played else +20,
//     Igralec.py:433-437).
// One warp per game replays the game from the hands as dealt + the exchange + the play history (so no per-step mask
// log is needed) and writes dy rows [48,54] (row t = play t; rows of unplayed slots are zero) plus the seat per row.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CTA) k_targets(Env e, const int* __restrict__ sel, u64 n_sel, float factor,
                                                 float* __restrict__ dy, uint8_t* __restrict__ seat_out,
                                                 uint8_t* __restrict__ rows_out) {
    const u32 lane = threadIdx.x & 31u;
    const u64 i = ((u64)blockIdx.x * CTA + threadIdx.x) >> 5;
    if (i >= n_sel) return;
    const u64 g = sel ? (u64)sel[i] : i;
    const u64 na = e.n_alloc;
    float* out = dy + i * (48u * 54u);
    warp_zero4(out, 48u * 54u, lane);
    for (u32 t = lane; t < 48; t += 32) { seat_out[i * 48u + t] = 0xFF; if (rows_out) rows_out[i * 48u + t] = 0; }
    __syncwarp();
    if (g >= e.n) return;
    const u64 meta = e.meta[g];
    if (mget(meta, M_PHASE, 2) != PH_DONE || ((meta >> M_ERR) & 1ull)) return;
    const u32 contract = mget(meta, M_CONTRACT, 4), decl = mget(meta, M_DECL, 2), plays = mget(meta, M_PLAYS, 6);
    const u32 grp = mget(meta, M_GROUP, 3);
    const bool klop = klop_rules(contract);
    const u64 order = e.torder[g];
    u64 h0 = e.hands0[g], h1 = e.hands0[na + g], h2 = e.hands0[2 * na + g], h3 = e.hands0[3 * na + g];
    if (grp != NO_GROUP) {                               // the exchange: group picked up, discards laid down
        const u64 nh = (sel4(h0, h1, h2, h3, decl) | talon_group_bits(order, talon_k(contract), grp)) & ~e.discard[g];
        h0 = decl == 0 ? nh : h0; h1 = decl == 1 ? nh : h1; h2 = decl == 2 ? nh : h2; h3 = decl == 3 ? nh : h3;
    }
    const u64 sc = e.scores[g];
    const u32 tricks_total = plays >> 2;
    const u32 extra = (grp != NO_GROUP ? 1u : 0u);
    for (u32 k = 0; k < tricks_total; k++) {
        u32 lead = 0;
        u64 bits = 0;
        u32 t24 = 0;
        u32 seats = 0;
#pragma unroll
        for (u32 j = 0; j < 4; j++) {
            const u32 t = 4 * k + j;
            const u32 hb = e.hist[(u64)t * na + g];
            const u32 s = hb >> 6, c = hb & 63u;
            if (j == 0) lead = c;
            const u64 hand = sel4(h0, h1, h2, h3, s);
            const u64 legal = legal_moves(hand, j != 0, lead, klop);
            // -70 on every illegal card of this row
            float* row = out + t * 54u;
            if (!((legal >> lane) & 1ull)) row[lane] = -70.f;
            if (lane + 32 < 54 && !((legal >> (lane + 32)) & 1ull)) row[lane + 32] = -70.f;
            if (lane == 0) {
                seat_out[i * 48u + t] = (uint8_t)s;
                if (rows_out) rows_out[i * 48u + t] = (uint8_t)padded_rows(t + extra + (contract == C_KLOP ? min(k, 6u) : 0u));
            }
            const u64 bit = 1ull << c;
            h0 ^= s == 0 ? bit : 0ull; h1 ^= s == 1 ? bit : 0ull; h2 ^= s == 2 ? bit : 0ull; h3 ^= s == 3 ? bit : 0ull;
            bits |= bit; t24 |= c << (6 * j); seats |= s << (2 * j);
        }
        if (contract == C_KLOP && k < 6) bits |= 1ull << ((order >> (6 * (5 - k))) & 63ull);
        const float v = (float)vrednost_stiha_bits(bits);
        const u32 wj = trick_winner(t24);
        __syncwarp();                                    // the -70 fills above precede the card entries below
        if (lane < 4) {
            const u32 t = 4 * k + lane;
            const u32 s = (seats >> (2 * lane)) & 3u, c = (t24 >> (6 * lane)) & 63u;
            float next;
            if (k + 1 < tricks_total) {                  // the seat's next_Q_max in the following trick
                next = 0.f;
                for (u32 jj = 0; jj < 4; jj++) {
                    const u32 t2 = 4 * (k + 1) + jj;
                    if ((u32)(e.hist[(u64)t2 * na + g] >> 6) == s) next = e.qmax_hist[(u64)t2 * na + g];
                }
            } else {                                     // final reward (Igralec.py:433-438)
                next = (float)(int16_t)(sc >> (16 * s));
                if (is_berac(contract) && s != decl) next = tricks_total == 12 ? -20.f : 20.f;
            }
            out[t * 54u + c] = (lane == wj ? v : -v) + factor * next;
        }
        __syncwarp();
    }
}

}  // namespace tk
