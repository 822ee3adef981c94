// Device-side Tarok rules on 64-bit card bitboards (bit i = card id i, Karta.v_id, Karta.py:19-23).
// Everything here is register arithmetic: popc / shifts / selects, no memory traffic.
// Reference behaviour incl. its quirks (SURVEY.md A.0) is cited per function.
#pragma once
#include <cstdint>

namespace tk {

using u64 = unsigned long long;
using u32 = unsigned int;

// ---- card constants (SURVEY.md A.1) --------------------------------------------------------
// id 0..7 KARA (1,2,3,4,J,C,Q,K), 8..15 SRCE, 16..23 PIK, 24..31 KRIZ, 32..53 TAROK I..XXII
constexpr u64 ALL54 = (1ull << 54) - 1;
constexpr u64 TAROKS = 0x3FFFFFull << 32;
constexpr u64 PAGAT = 1ull << 32;
constexpr u64 KINGS = (1ull << 7) | (1ull << 15) | (1ull << 23) | (1ull << 31);
constexpr u64 QUEENS = KINGS >> 1;
constexpr u64 CAVALS = KINGS >> 2;
constexpr u64 JACKS = KINGS >> 3;
constexpr u64 TRULA = (1ull << 32) | (1ull << 52) | (1ull << 53);
// Roka.mozno_zalozit (Roka.py:23-27) with the buggy Karta.vrednost (Karta.py:10-16):
// suit ranks 1..7 and taroks II..VII may be laid down (Q8).
constexpr u64 DISCARDABLE = 0x7F7F7F7Full | (0x3Full << 33);

// ---- contract codes = Tip_igre value / 10 (Tip_igre.py:5-15) ---------------------------------
enum : int { C_NAPREJ = -1, C_KLOP = 0, C_TRI, C_DVE, C_ENA, C_SOLO_TRI, C_SOLO_DVE, C_SOLO_ENA,
             C_BERAC, C_SOLO_BREZ, C_ODPRTI_BERAC, C_NONE = 15 };
constexpr u32 NO_KING = 7;
constexpr u32 NO_GROUP = 7;

__device__ __forceinline__ bool is_navadna(u32 c) { return (c >= C_TRI && c <= C_SOLO_ENA) || c == C_SOLO_BREZ; }
__device__ __forceinline__ bool is_king_game(u32 c) { return c >= C_TRI && c <= C_ENA; }
__device__ __forceinline__ bool is_berac(u32 c) { return c == C_BERAC || c == C_ODPRTI_BERAC; }
// Klop.mozne_karte is inherited by Berac (Berac.py:4)
__device__ __forceinline__ bool klop_rules(u32 c) { return c == C_KLOP || is_berac(c); }
// st_kart_za_menjat / korak (Navadna_igra.py:36-58); 0 = no exchange.  Two bits per contract code in one constant:
// Tri / Solo_tri 3, Dve / Solo_dve 2, Ena / Solo_ena 1, everything else (incl. code 15 = none) 0.
__device__ __forceinline__ u32 talon_k(u32 c) { return (0x1B6Cu >> (2u * (c & 15u))) & 3u; }

// ---- meta word layout -----------------------------------------------------------------------
// Fields never straddle the 32-bit halves, so every update is 32-bit integer work.
//  low word : 0-3 contract code (15 = none)   4-5 declarer   6-8 king suit (7 = none)   9-12 ekipa seat mask
//             13-14 leader (zacne)   15-16 pos = cards in the current trick   17-20 tricks completed
//             21-22 last trick winner   23 trick-just-completed   24-25 phase (0 dealt 1 await-exchange
//             2 playing 3 finished)   26 error   27-29 chosen talon group (7 none)
//             30 Klop-family rules (Klop / Berac / Odprti_berac: pagat restriction), cached from the contract code
//  high word: 32-55 trick cards, 6 bits each, play order   56-61 plays made (0..48)   62 scored/pad
constexpr int M_CONTRACT = 0, M_DECL = 4, M_KING = 6, M_TEAM = 9, M_LEADER = 13, M_POS = 15,
              M_TRICKS = 17, M_WINNER = 21, M_TRICKDONE = 23, M_PHASE = 24, M_ERR = 26, M_GROUP = 27, M_KLOPFAM = 30,
              M_TRICK = 32, M_PLAYS = 56, M_SCORED = 62;
enum : u32 { PH_DEALT = 0, PH_EXCHANGE = 1, PH_PLAY = 2, PH_DONE = 3 };

__device__ __forceinline__ u32 mget(u64 m, int sh, u32 bits) { return (u32)(m >> sh) & ((1u << bits) - 1u); }
__device__ __forceinline__ u64 mset(u64 m, int sh, u32 bits, u32 v) {
    return (m & ~((u64)((1u << bits) - 1u) << sh)) | ((u64)v << sh);
}
__device__ __forceinline__ u64 meta_fresh() {
    return ((u64)C_NONE << M_CONTRACT) | ((u64)NO_KING << M_KING) | ((u64)NO_GROUP << M_GROUP);
}
__device__ __forceinline__ u64 meta_pad() { return meta_fresh() | ((u64)PH_DONE << M_PHASE) | (1ull << M_SCORED); }

// ---- small helpers --------------------------------------------------------------------------
__device__ __forceinline__ u64 sel4(u64 a, u64 b, u64 c, u64 d, u32 i) {
    u64 lo = (i & 1) ? b : a, hi = (i & 1) ? d : c;
    return (i & 2) ? hi : lo;
}
// r-th (0-based) lowest set bit of m; r < popc(m).  Binary descent on one 32-bit half.
__device__ __forceinline__ u32 nth_set_bit(u64 m, u32 r) {
    const u32 lo = (u32)m, hi = (u32)(m >> 32);
    const u32 cl = __popc(lo);
    const bool up = r >= cl;
    u32 w = up ? hi : lo;
    r -= up ? cl : 0u;
    u32 pos = up ? 32u : 0u, c;
    c = __popc(w & 0xFFFFu); if (r >= c) { r -= c; w >>= 16; pos += 16; }
    c = __popc(w & 0xFFu);   if (r >= c) { r -= c; w >>= 8;  pos += 8; }
    c = __popc(w & 0xFu);    if (r >= c) { r -= c; w >>= 4;  pos += 4; }
    c = __popc(w & 0x3u);    if (r >= c) { r -= c; w >>= 2;  pos += 2; }
    pos += (r >= (w & 1u)) ? 1u : 0u;
    return pos;
}
// The last three levels of that descent as a table: SELECT8[8 * v + r] = position of the r-th set bit of the byte v
// (r < popc(v); 0 otherwise).  2 KB, built at compile time; the hot kernels copy it into shared memory once per CTA
// (select8_to_shared) and finish the descent with one LDS instead of ~20 integer instructions -- the integer ALU pipe is
// what bounds play_step.
struct Select8 { uint8_t v[2048]; };
constexpr Select8 make_select8() {
    Select8 t{};
    for (int v = 0; v < 256; v++) {
        int r = 0;
        for (int b = 0; b < 8; b++)
            if ((v >> b) & 1) t.v[8 * v + r++] = (uint8_t)b;
    }
    return t;
}
__device__ const Select8 SELECT8 = make_select8();
constexpr int SELECT8_SMEM = 2048 + 16;                   // the slack keeps a stray index (r up to 11 on a garbage lane) inside
// All threads of the CTA (CTA == 256: 8 bytes each), then a barrier before the first lookup.
__device__ __forceinline__ uint2 select8_fetch() { return reinterpret_cast<const uint2*>(SELECT8.v)[threadIdx.x]; }
__device__ __forceinline__ void select8_store(uint8_t* sh, uint2 mine) {
    reinterpret_cast<uint2*>(sh)[threadIdx.x] = mine;
    if (threadIdx.x < 4) reinterpret_cast<u32*>(sh + 2048)[threadIdx.x] = 0u;
}
__device__ __forceinline__ void select8_to_shared(uint8_t* sh) { select8_store(sh, select8_fetch()); }
__device__ __forceinline__ u32 nth_set_bit_lut(u64 m, u32 r, const uint8_t* __restrict__ sel8) {
    const u32 lo = (u32)m, hi = (u32)(m >> 32);
    const u32 cl = __popc(lo);
    const bool up = r >= cl;
    u32 w = up ? hi : lo;
    r -= up ? cl : 0u;
    u32 pos = up ? 32u : 0u, c;
    c = __popc(w & 0xFFFFu); if (r >= c) { r -= c; w >>= 16; pos += 16; }
    c = __popc(w & 0xFFu);   if (r >= c) { r -= c; w >>= 8;  pos += 8; }
    return pos + sel8[(w & 0xFFu) * 8u + r];
}
__device__ __forceinline__ u64 suit_mask_of(u32 card) {
    return card >= 32 ? TAROKS : (0xFFull << (card & 24u));
}

// ---- legal moves ----------------------------------------------------------------------------
// Navadna_igra.mozne_karte (Navadna_igra.py:158-168): follow suit, else must trump, else anything.
// Klop.mozne_karte (Klop.py:96-133), *effective* behaviour (Q1): the overtake filter is computed and
// dropped (Klop.py:104), leaving the same set minus the pagat whenever more than one card is legal.
// Written on the 32-bit halves: the low word holds the four suits, the high word only taroks.
__device__ __forceinline__ u64 legal_moves(u64 hand, bool has_lead, u32 lead, bool klop) {
    const u32 lo = (u32)hand, hi = (u32)(hand >> 32);
    u32 mlo = lo, mhi = hi;
    if (has_lead) {
        const u32 f = lead < 32u ? (lo & (0xFFu << (lead & 24u))) : 0u;   // cards of the led suit (taroks: via hi)
        mlo = f ? f : (hi ? 0u : lo);
        mhi = f ? 0u : hi;
    }
    if (klop) {
        const u32 rest = mhi & ~1u;                                        // without the pagat (tarok I = bit 32)
        if (mlo | rest) mhi = rest;
    }
    return ((u64)mhi << 32) | mlo;
}

// pobere_stih / primerjaj_karti (Navadna_igra.py:143-156, Klop.py:81-94): scan cards 1..3 against the
// current best: same suit and higher rank, or a tarok over a non-tarok.  No trula/pagat rule (Q3).
// Branch-free form: only a tarok or a card of the led suit can ever be "best", and among those the larger id wins
// (taroks are ids 32..53, above every suit card; within a suit a larger id is a higher rank), so the winner is the arg-max
// of key_i = eligible_i ? ((c_i + 1) << 2 | i) : 0.  Same suit as the lead <=> (c ^ lead) < 8 for a suit lead; for a tarok
// lead that test only ever adds taroks.  Checked against the sequential scan on all 54*53*52*51 ordered tricks
// (tests/test_closed_forms.py).
__device__ __forceinline__ u32 trick_winner(u32 t24) {
    const u32 lead = t24 & 63u;
    u32 m = ((lead + 1u) << 2);
#pragma unroll
    for (u32 i = 1; i < 4; i++) {
        const u32 c = (t24 >> (6u * i)) & 63u;
        const bool eligible = c >= 32u || (c ^ lead) < 8u;
        m = max(m, eligible ? (((c + 1u) << 2) | i) : 0u);
    }
    return m & 3u;
}

// Roka.prestej (Roka.py:55-98): groups of three, sum-2; a remainder of one or two cards, sum-1 (Q10).
// Order independent: sum(points) - 2*floor(n/3) - [n%3 != 0].
__device__ __forceinline__ int prestej(u64 s) {
    int n = __popcll(s);
    int pts = n + __popcll(s & JACKS) + 2 * __popcll(s & CAVALS) + 3 * __popcll(s & QUEENS)
            + 4 * __popcll(s & (KINGS | TRULA));
    return pts - 2 * (n / 3) - ((n % 3) != 0);
}
__device__ __forceinline__ int prestej_pn(int pts, int n) { return pts - 2 * (n / 3) - ((n % 3) != 0); }
// value of one trick for per-trick rewards: Roka.vrednost_stiha on 4 or 5 cards = sum - 2 (Roka.py:92-95)
__device__ __forceinline__ int vrednost_stiha_bits(u64 s) {
    int n = __popcll(s);
    int pts = n + __popcll(s & JACKS) + 2 * __popcll(s & CAVALS) + 3 * __popcll(s & QUEENS)
            + 4 * __popcll(s & (KINGS | TRULA));
    return pts - ((n == 1 || n == 2) ? 1 : 2);
}

// ---- auction ----------------------------------------------------------------------------------
// Igralec.licitiram filter (Igralec.py:58-74).  obv < -1 encodes "obvezno is None".
constexpr int OBV_NONE = -2;
__device__ __forceinline__ int bid_filter(int want, int min_igra, int obv, bool pred) {
    bool ok = pred ? (want >= min_igra) : (want > min_igra);
    return ok ? want : (obv == OBV_NONE ? (int)C_NAPREJ : obv);
}

// Igra.licitacija (Igra.py:75-114) as a state machine over a bidder functor
//   int Want::operator()(int seat, int call_index)   -> the Tip code the seat wants at this call;
//   bool Want::fixed(int seat)                        -> the seat's bidding semantics, per seat:
// fixed = Nevronski_igralec: the first answer is kept and overwritten by every returned value (Igralec.py:295-304);
// otherwise (Bot_igralec, Igralec.py:151) every call asks afresh.
template <class Want>
__device__ __forceinline__ void licitacija(Want& want, int& declarer, int& contract) {
    int intent[4] = {C_NONE, C_NONE, C_NONE, C_NONE};
    int calls = 0;
    auto call = [&](int seat, int mn, int obv, bool pred) -> int {
        const bool fixed = want.fixed(seat);
        int w;
        if (fixed) {
            if (intent[seat] == C_NONE) intent[seat] = want(seat, calls);
            w = intent[seat];
        } else {
            w = want(seat, calls);
        }
        calls++;
        int r = bid_filter(w, mn, obv, pred);
        if (fixed) intent[seat] = r;
        return r;
    };
    u32 lic = 0;
    int mx = C_TRI;
#pragma unroll
    for (int s = 1; s < 4; s++) {
        int r = call(s, mx, OBV_NONE, false);
        if (r != C_NAPREJ) lic |= 1u << s;
        mx = max(mx, r);
    }
    if (mx == C_TRI) {                                   // nobody bid: forehand plays own game or Klop
        declarer = 0;
        contract = call(0, C_NAPREJ, C_KLOP, false);
        return;
    }
    {
        int r = call(0, mx, OBV_NONE, true);             // forehand has priority (prednost)
        if (r != C_NAPREJ) lic |= 1u;
        mx = max(mx, r);
    }
    int holder = __ffs(lic) - 1;                         // min(lic)
    for (int guard = 0; __popc(lic) != 1 && guard < 32; guard++) {
        u32 nl = 0;
#pragma unroll
        for (int j = 1; j <= 4; j++) {                   // sorted keys with seat 0 moved last
            int k = j & 3;
            if (!((lic >> k) & 1u)) continue;
            int r = (k == holder) ? call(k, mx, mx, false) : call(k, mx, OBV_NONE, false);
            if (r != C_NAPREJ) { nl |= 1u << k; holder = k; mx = r; }
        }
        lic = nl;
    }
    declarer = holder;
    contract = mx;
}

// Nevronski_igralec.index2igra (Igralec.py:717-745) + two raw extras (18 Odprti_berac, 19 Klop); idx <= 19 (callers reject
// larger indices: tarok_auction makes them error games)
__device__ __forceinline__ void index2igra(u32 idx, int& tip, u32& suit) {
    suit = NO_KING;
    if (idx == 0) tip = C_NAPREJ;
    else if (idx <= 12) { tip = C_TRI + (int)((idx - 1) >> 2); suit = (idx - 1) & 3u; }
    else if (idx <= 15) tip = C_SOLO_TRI + (int)(idx - 13);
    else if (idx == 16) tip = C_BERAC;
    else if (idx == 17) tip = C_SOLO_BREZ;
    else if (idx == 18) tip = C_ODPRTI_BERAC;
    else tip = C_KLOP;
}

// ---- contract start ---------------------------------------------------------------------------
// Igra.start dispatch (Igra.py:38-58) + constructors: Navadna_igra.__init__ teams from the
// pre-exchange hands (Navadna_igra.py:20-30, Q9), leader 0 (Navadna_igra.py:70, Klop.py:26) or the
// declarer for Berac (Berac.py:15, Q11).  Returns the new meta word.
__device__ __forceinline__ u64 begin_contract(u64 meta, u32 contract, u32 declarer, u32 king,
                                              u64 h0, u64 h1, u64 h2, u64 h3) {
    bool bad = contract > C_ODPRTI_BERAC || declarer > 3;
    if (contract == C_KLOP) declarer = 0;
    u32 team = 0, leader = 0, phase = PH_PLAY;
    if (!bad && is_king_game(contract)) {
        if (king > 3) bad = true;                        // assert barva_kralja != TAROK (Navadna_igra.py:21)
        u64 kb = 1ull << ((king & 3u) * 8 + 7);
        team = (1u << declarer) | ((h0 & kb) ? 1u : 0u) | ((h1 & kb) ? 2u : 0u) | ((h2 & kb) ? 4u : 0u)
             | ((h3 & kb) ? 8u : 0u);
    } else {
        king = NO_KING;
        if (!bad && is_navadna(contract)) team = 1u << declarer;
    }
    if (!bad) {
        if (is_berac(contract)) leader = declarer;
        if (talon_k(contract) != 0) phase = PH_EXCHANGE;
    }
    // every field this function owns sits in the low word; the rest of the word (trick leader / position / counters,
    // error bit, chosen group) is kept
    constexpr u32 OWNED = (15u << M_CONTRACT) | (3u << M_DECL) | (7u << M_KING) | (15u << M_TEAM) | (3u << M_LEADER)
                        | (3u << M_PHASE) | (1u << M_KLOPFAM);
    const u32 lo = ((u32)meta & ~OWNED) | ((bad ? (u32)C_NONE : contract) << M_CONTRACT) | ((declarer & 3u) << M_DECL)
                 | ((king & 7u) << M_KING) | (team << M_TEAM) | (leader << M_LEADER) | ((bad ? (u32)PH_DONE : phase) << M_PHASE)
                 | (((!bad && klop_rules(contract)) ? 1u : 0u) << M_KLOPFAM);
    meta = (meta & 0xFFFFFFFF00000000ull) | lo;
    if (bad) meta |= 1ull << M_ERR;
    return meta;
}

// ---- talon exchange -----------------------------------------------------------------------------
// Group g of Navadna_igra.odpri_talon (Navadna_igra.py:36-44): consecutive slices of the ordered talon.
__device__ __forceinline__ u64 talon_group_bits(u64 order, u32 k, u32 g) {
    const u64 w = order >> (6u * g * k);                 // the group's ids are the next k six-bit fields
    u64 b = 1ull << (w & 63ull);
    if (k > 1) b |= 1ull << ((w >> 6) & 63ull);
    if (k > 2) b |= 1ull << ((w >> 12) & 63ull);
    return b;
}

// ---- one card play ------------------------------------------------------------------------------
// krog body (Navadna_igra.py:115-141 / Klop.py:47-79) for the seat to move.  `hand` is the mover's
// hand.  On trick completion reports the winner seat and the bitboard that goes to its pile; Klop adds
// the talon card popped from the END of the ordered talon in tricks 1..6 (Klop.py:67-71, Q4), which
// never competes for the trick (Klop.py:81-86).  Berac stops when the declarer takes a trick
// (Berac.py:33-39, Q12).
struct PlayResult {
    bool trick_done;
    u32 winner_rel;   // the winner's index in the trick's play order (= its hand slot)
    u32 winner;       // absolute seat
    u64 pile_bits;    // cards the winner collects
    u64 talon_clear;  // Klop: talon bit consumed
};

// CHECK = validate the card against the legal set (externally supplied actions); the in-kernel random
// players pick from the legal set by construction and skip it.
// POS >= 0: the caller knows (and has checked) that the game is at position POS of its trick -- lock-step batches --
// so the trick-position arithmetic and the trick-end branch fold at compile time; POS = -1 reads it from meta.
// BITS = also produce the bitboard the winner collects (+ the Klop talon card); the stepwise kernels do not need it:
// they append (cards, winner) to the trick log and the piles are materialised at scoring time (trick_bits below).
template <bool CHECK, int POS = -1, bool BITS = true>
__device__ __forceinline__ u64 play_card(u64 meta, u64& hand, u32 card, u64 talon, u64 talon_order,
                                         PlayResult& out) {
    out.trick_done = false; out.winner = 0; out.winner_rel = 0; out.pile_bits = 0; out.talon_clear = 0;
    u32 lo = (u32)meta, hi = (u32)(meta >> 32);
    const u32 contract = lo & 15u;
    const u32 pos = POS >= 0 ? (u32)POS : ((lo >> M_POS) & 3u);
    const u64 bit = (!CHECK || card < 54) ? (1ull << (card & 63u)) : 0ull;   // in-kernel picks are in range by construction
    if (CHECK) {
        u64 legal = legal_moves(hand, pos != 0, hi & 63u, (lo >> M_KLOPFAM) & 1u);
        if (!(legal & bit)) {                             // 'Karte ne mores igarti' (Navadna_igra.py:125-126)
            lo |= (1u << M_ERR) | (PH_DONE << M_PHASE);
            return ((u64)hi << 32) | lo;
        }
    }
    hand ^= bit;
    const u32 tr = (pos ? (hi & 0xFFFFFFu) : 0u) | (card << (6u * pos));
    hi = tr | ((hi & 0xFF000000u) + (1u << (M_PLAYS - 32)));           // trick cards | plays + 1 (| scored bit)
    if (pos < 3) {
        lo = (lo & ~(1u << M_TRICKDONE)) + (1u << M_POS);
        return ((u64)hi << 32) | lo;
    }
    // trick complete
    const u32 tricks = (lo >> M_TRICKS) & 15u;
    const u32 wr = trick_winner(tr);
    const u32 w = (((lo >> M_LEADER) & 3u) + wr) & 3u;
    out.winner_rel = wr;
    if (BITS) {
        u64 bits = (1ull << (tr & 63u)) | (1ull << ((tr >> 6) & 63u)) | (1ull << ((tr >> 12) & 63u)) | (1ull << (tr >> 18));
        if (contract == C_KLOP && tricks < 6) {
            u64 tc = 1ull << ((talon_order >> (6 * (5 - tricks))) & 63ull);
            out.talon_clear = tc & talon;
            bits |= out.talon_clear;
        }
        out.pile_bits = bits;
    }
    out.trick_done = true; out.winner = w;
    // Berac (the Klop-family contracts other than Klop itself) stops when the declarer takes a trick
    const bool fin = tricks == 11 || (((lo >> M_KLOPFAM) & 1u) && contract != C_KLOP && w == ((lo >> M_DECL) & 3u));
    constexpr u32 CLEAR = (3u << M_LEADER) | (3u << M_POS) | (15u << M_TRICKS) | (3u << M_WINNER) | (1u << M_TRICKDONE)
                        | (3u << M_PHASE);
    lo = (lo & ~CLEAR) | (w << M_LEADER) | ((tricks + 1u) << M_TRICKS) | (w << M_WINNER) | (1u << M_TRICKDONE)
       | ((fin ? (u32)PH_DONE : (u32)PH_PLAY) << M_PHASE);              // the finished trick stays visible in hi
    return ((u64)hi << 32) | lo;
}

// Card points of the four cards of a trick (Roka.vrednost_stiha's per-card values, Roka.py:76-91: suit ranks 1-4 -> 1,
// J 2, C 3, Q 4, K 5; taroks 1, trula 5), computed on the packed 4 x 6-bit card ids at once (no per-card loop):
// bit 5 of a field = tarok, bit 2 of a suit card = J or higher, and its low two bits + 1 = the extra points.
// Checked against the per-card table on all 54^4 tuples (tests/test_closed_forms.py).
__device__ __forceinline__ u32 trick_points(u32 f) {
    const u32 B5 = 0x820820u;                                        // bit 5 of every field
    const u32 hr = ~f & (f << 3) & B5;                               // suit card with rank >= J
    const u32 v = ((f & 0x0C30C3u) + 0x041041u) & ((hr >> 5) * 7u);  // 1..4 extra for J, C, Q, K
    const u32 a = f & (f << 1) & (f << 3);                           // bit 5: ids 52, 53 (mond, skis)
    const u32 nz = (f & 0x7DF7DFu) + 0x7DF7DFu;                      // bit 5 set iff the low five bits are not all zero
    const u32 tr = f & (a | ~nz) & B5;                               // trula: id 32 (pagat) | 52 | 53
    return 4u + (((v * 0x041041u) >> 18) & 0x3Fu) + 4u * (u32)__popc(tr);
}
__device__ __forceinline__ u32 card_points1(u32 c) {                 // one card
    return c >= 32u ? ((c == 32u || c >= 52u) ? 5u : 1u) : ((c & 4u) ? (c & 7u) - 2u : 1u);
}
// Does the trick (4 x 6-bit ids) contain card `id`?
__device__ __forceinline__ bool trick_has(u32 f, u32 id) {
    const u32 x = (f & 0xFFFFFFu) ^ (id * 0x041041u);
    const u32 z = ((x & 0x7DF7DFu) + 0x7DF7DFu) | x;                 // bit 5 of a field set iff the field is non-zero
    return (~z & 0x820820u) != 0u;
}
// Trick-log entry: the four cards in play order (bits 0-23) | trick_points (24-28) | bit 29: the trick contains the CALLED
// king (king games only; Navadna_igra.py:87 asks whether that card ended in the declarer's pile) | winner seat (30-31, so
// that scoring reads it with one shift).
__device__ __forceinline__ u32 log_entry(u32 t24, u32 winner, u32 meta_lo) {
    const u32 king = (meta_lo >> M_KING) & 7u;
    const u32 kf = (king != NO_KING && trick_has(t24, king * 8u + 7u)) ? (1u << 29) : 0u;
    return t24 | (trick_points(t24) << 24) | kf | (winner << 30);
}
// Trick-log entry, continued.  The bitboard the winner collected in
// trick k: its four cards, plus in Klop the talon card popped from the END of the ordered talon in tricks 1..6
// (Klop.py:67-71, Q4), which is also returned in `talon_card`.
__device__ __forceinline__ u64 trick_bits(u32 entry, u32 k, bool is_klop, u64 talon_order, u64& talon_card) {
    u64 bits = (1ull << (entry & 63u)) | (1ull << ((entry >> 6) & 63u)) | (1ull << ((entry >> 12) & 63u))
             | (1ull << ((entry >> 18) & 63u));
    talon_card = 0;
    if (is_klop && k < 6) { talon_card = 1ull << ((talon_order >> (6 * (5 - k))) & 63ull); bits |= talon_card; }
    return bits;
}

// Legal mask of the seat to move given the (already updated) meta and that seat's hand.
__device__ __forceinline__ u64 mask_for_mover(u64 meta, u64 hand) {
    if (mget(meta, M_PHASE, 2) != PH_PLAY) return 0ull;
    u32 pos = mget(meta, M_POS, 2);
    return legal_moves(hand, pos != 0, mget(meta, M_TRICK, 6), ((u32)meta >> M_KLOPFAM) & 1u);
}
__device__ __forceinline__ u32 mover_of(u64 meta) { const u32 lo = (u32)meta; return ((lo >> M_LEADER) + (lo >> M_POS)) & 3u; }

// ---- scoring --------------------------------------------------------------------------------------
// Epilogues: Navadna_igra.start (Navadna_igra.py:80-113, Q6/Q7), Klop.start (Klop.py:36-45, Q5),
// Berac.start (Berac.py:33-44).  Returns the four scores packed as int16 x4 (seat 0 in the low half).
__device__ __forceinline__ u64 pack_scores(int s0, int s1, int s2, int s3) {
    return (u64)(uint16_t)s0 | ((u64)(uint16_t)s1 << 16) | ((u64)(uint16_t)s2 << 32) | ((u64)(uint16_t)s3 << 48);
}

// Navadna_igra.start epilogue from the team's pile union `tp` and the declarer's own pile `pd` (Navadna_igra.py:80-113).
__device__ __forceinline__ u64 score_navadna(u64 meta, u64 tp, u64 pd, u64 talon) {
    const u32 contract = mget(meta, M_CONTRACT, 4), team = mget(meta, M_TEAM, 4), king = mget(meta, M_KING, 3);
    const bool to_team = contract != C_SOLO_BREZ && __popc(team) == 1 && king != NO_KING
                      && (pd & (1ull << ((king & 3u) * 8 + 7)));
    if (to_team) tp |= talon;                             // leftover talon to a lone declarer who took the called king (Q7)
    const int v = prestej(tp);
    const int r = v - 35 + 2;                             // 5*round((v-35)/5): no ties for integers
    const int q = (r >= 0 ? r / 5 : -((-r + 4) / 5)) * 5; // floor division
    const int val = (v > 35 ? 10 * (int)contract : -10 * (int)contract) + q;
    return pack_scores((team & 1u) ? val : 0, (team & 2u) ? val : 0, (team & 4u) ? val : 0, (team & 8u) ? val : 0);
}

// The same epilogue from the team's card points and card count (prestej is order independent).
__device__ __forceinline__ u64 score_navadna_v(u64 meta, int v) {
    const u32 contract = mget(meta, M_CONTRACT, 4), team = mget(meta, M_TEAM, 4);
    const int r = v - 35 + 2;
    const int q = (r >= 0 ? r / 5 : -((-r + 4) / 5)) * 5;
    const int val = (v > 35 ? 10 * (int)contract : -10 * (int)contract) + q;
    return pack_scores((team & 1u) ? val : 0, (team & 2u) ? val : 0, (team & 4u) ? val : 0, (team & 8u) ? val : 0);
}

// Klop.start epilogue (Klop.py:36-45): minus the own points; if anybody has more than 35 everybody writes 0 (Q5).
__device__ __forceinline__ u64 score_klop(u64 p0, u64 p1, u64 p2, u64 p3) {
    const int a = prestej(p0), b = prestej(p1), c = prestej(p2), d = prestej(p3);
    const bool any = a > 35 || b > 35 || c > 35 || d > 35;
    return pack_scores(any ? 0 : -a, any ? 0 : -b, any ? 0 : -c, any ? 0 : -d);
}

// Berac.start (Berac.py:33-44): -70/-90 as soon as the declarer took a trick, else +70/+90; the others 0.
__device__ __forceinline__ u64 score_berac(u64 meta, bool declarer_took_a_trick) {
    const u32 decl = mget(meta, M_DECL, 2);
    const int v = mget(meta, M_CONTRACT, 4) == C_ODPRTI_BERAC ? 90 : 70;
    const int x = declarer_took_a_trick ? -v : v;
    return pack_scores(decl == 0 ? x : 0, decl == 1 ? x : 0, decl == 2 ? x : 0, decl == 3 ? x : 0);
}

__device__ __forceinline__ u64 score_game(u64 meta, u64 p0, u64 p1, u64 p2, u64 p3, u64 talon) {
    const u32 contract = mget(meta, M_CONTRACT, 4);
    const u32 decl = mget(meta, M_DECL, 2);
    if (is_navadna(contract)) {
        const u32 team = mget(meta, M_TEAM, 4);
        const u64 tp = ((team & 1u) ? p0 : 0) | ((team & 2u) ? p1 : 0) | ((team & 4u) ? p2 : 0) | ((team & 8u) ? p3 : 0);
        return score_navadna(meta, tp, sel4(p0, p1, p2, p3, decl), talon);
    }
    if (contract == C_KLOP) return score_klop(p0, p1, p2, p3);
    if (is_berac(contract)) return score_berac(meta, sel4(p0, p1, p2, p3, decl) != 0);   // no exchange in Berac
    return 0;
}

}  // namespace tk
