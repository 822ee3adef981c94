/* TEST INFRASTRUCTURE ONLY -- synthetic-input generator + uniform-random players for the oracle.
 *
 * NOT reference behaviour: the reference deals with random.shuffle on MT19937 and its bots draw
 * from the random/numpy global streams (Igra.py:67, Igralec.py:151,156,159,166), none of which is
 * seeded (main.py:174 is commented out).  Parity is therefore by deal/action injection, and this
 * file restates -- independently, in scalar C on top of tarok_oracle.c's list-based engine -- the
 * counter-based Philox4x32-10 input generator that the CUDA path uses (DESIGN.md "Synthetic
 * inputs"), so whole rollouts can be compared at full size on the GPU box:
 *
 *   word(gid, stream, idx)  = philox4x32_10(key = seed, ctr = {gid.lo, gid.hi, stream | attempt<<16, idx>>2})[idx&3]
 *   draw(gid, stream, idx, n) = Lemire multiply-shift with rejection on word(...) -> uniform in [0,n)
 *   batched draws: k exact draws with bounds n_1..n_k from ONE word x: r_i = hi32(x * n_i), x = lo32(x * n_i); the tuple is
 *     accepted iff the final x >= 2^32 mod (n_1 * ... * n_k) (Lemire's method for the product bound, read digit by digit),
 *     else the word is redrawn with attempt = 1, 2, ...
 *   streams: 0 deal, 1 bids, 4 play, 5 setup (forced contract / declarer / king, exchange), 6 play retry, 7 deal retry
 *   play draws (n <= 12) use 16-bit lanes: one Philox block per (game pair = gid>>1, trick) holds eight
 *   16-bit values, lane = (gid&1)*4 + play-in-trick; 16-bit Lemire, rejected sliver -> 32-bit draw on stream 6
 *
 * It doubles as bench.py's CPU baseline ("port": OpenMP over games).
 */
#include <string.h>
#include <stdint.h>
#include "tarok_oracle.h"

#define PH_M0 0xD2511F53u
#define PH_M1 0xCD9E8D57u
#define PH_W0 0x9E3779B9u
#define PH_W1 0xBB67AE85u

enum { ST_DEAL = 0, ST_BID = 1, ST_KING = 2, ST_EXCH = 3, ST_PLAY = 4, ST_FORCE = 5, ST_PLAY_RETRY = 6, ST_DEAL_RETRY = 7 };
enum { MODE_NAVADNA_MIX = 16, MODE_AUCTION_UNIFORM = 17, MODE_AUCTION_BOT = 18 };

void syn_philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
    for (int r = 0; r < 10; r++) {
        uint64_t p0 = (uint64_t)PH_M0 * c[0];
        uint64_t p1 = (uint64_t)PH_M1 * c[2];
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
        k0 += PH_W0; k1 += PH_W1;
    }
}

uint32_t syn_draw(uint64_t seed, uint64_t gid, uint32_t stream, uint32_t idx, uint32_t n) {
    for (uint32_t attempt = 0;; attempt++) {
        uint32_t c[4] = { (uint32_t)gid, (uint32_t)(gid >> 32), stream | (attempt << 16), idx >> 2 };
        syn_philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
        uint64_t m = (uint64_t)c[idx & 3] * n;
        uint32_t lo = (uint32_t)m;
        if (lo >= n) return (uint32_t)(m >> 32);
        uint32_t t = (0u - n) % n;
        if (lo >= t) return (uint32_t)(m >> 32);
    }
}


static uint32_t bdraw(uint32_t* x, uint32_t n) {
    uint64_t m = (uint64_t)(*x) * n;
    *x = (uint32_t)m;
    return (uint32_t)(m >> 32);
}

/* k batched draws from word `word` of (gid, stream): attempt 0 reads the stream's own block, a rejected word is redrawn
   from (retry_stream | attempt << 16) with attempt = 1, 2, ... */
static void syn_bdraws(uint64_t seed, uint64_t gid, uint32_t stream, uint32_t retry_stream, uint32_t word,
                       const uint32_t* n, int k, uint32_t* r) {
    for (uint32_t attempt = 0;; attempt++) {
        uint32_t c[4] = { (uint32_t)gid, (uint32_t)(gid >> 32), attempt ? (retry_stream | (attempt << 16)) : stream, word >> 2 };
        syn_philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
        uint32_t x = c[word & 3], prod = 1;
        for (int i = 0; i < k; i++) { r[i] = bdraw(&x, n[i]); prod *= n[i]; }
        if (x >= (uint32_t)((1ull << 32) % prod)) return;
    }
}

/* Uniform deal: card c = 0..53 goes to a uniformly random free slot among the 54-c left; slots
   are exchangeable inside a pile, so this is a walk over the remaining capacities of the piles
   (seat 0..3: 12 each, then the talon: 6).  The 53 draws are batched: words 0..5 of the deal stream carry
   three cards each (cards 0..17), words 6..13 four each (cards 18..49), word 14 cards 50..52; card 53 takes the
   last slot.  The ORDER of the six talon cards (it matters: Navadna_igra.py:44, Klop.py:69) is a uniform
   permutation decoded from word 15 (32-bit Lemire, n = 720, Lehmer code over the talon ids in ascending order).
   Exported as the permutation Igra.razdeli would have consumed: seat slices ascending by id, then the ordered talon. */
void syn_deal(uint64_t seed, uint64_t gid, uint8_t perm[54]) {
    int cap[4] = { 12, 12, 12, 12 }, fill[4] = { 0, 0, 0, 0 };
    uint8_t tal[6];
    int nt = 0;
    uint32_t draws[54];
    for (int w = 0; w < 15; w++) {
        int c0 = w < 6 ? 3 * w : w < 14 ? 18 + 4 * (w - 6) : 50;
        int nc = (w < 6 || w == 14) ? 3 : 4;
        uint32_t n[4];
        for (int i = 0; i < nc; i++) n[i] = (uint32_t)(54 - (c0 + i));
        syn_bdraws(seed, gid, ST_DEAL, ST_DEAL_RETRY, (uint32_t)w, n, nc, draws + c0);
    }
    draws[53] = 0;
    for (int c = 0; c < 54; c++) {
        uint32_t r = draws[c];
        int s;
        for (s = 0; s < 4; s++) {
            if (r < (uint32_t)cap[s]) break;
            r -= (uint32_t)cap[s];
        }
        if (s < 4) { perm[12 * s + fill[s]++] = (uint8_t)c; cap[s]--; }
        else tal[nt++] = (uint8_t)c;
    }
    uint32_t cw[4] = { (uint32_t)gid, (uint32_t)(gid >> 32), ST_DEAL, 3 };
    syn_philox4x32_10(cw, (uint32_t)seed, (uint32_t)(seed >> 32));
    uint64_t mm = (uint64_t)cw[3] * 720u;
    uint32_t L = (uint32_t)(mm >> 32);
    if ((uint32_t)mm < 256u) L = syn_draw(seed, gid, ST_DEAL_RETRY, 54, 720);     /* 2^32 % 720 = 256 */
    static const uint32_t fact[6] = { 120, 24, 6, 2, 1, 1 };
    int left = 6;
    for (int i = 0; i < 6; i++) {
        uint32_t d = L / fact[i];
        L -= d * fact[i];
        perm[48 + i] = tal[d];
        memmove(tal + d, tal + d + 1, (size_t)(left - (int)d - 1));
        left--;
    }
}

/* Nevronski_igralec.index2igra (Igralec.py:717-745): 0 (Naprej,-), 1-4 (Tri,suit), 5-8 (Dve,suit),
   9-12 (Ena,suit), 13 Solo_tri, 14 Solo_dve, 15 Solo_ena, 16 Berac, 17 Solo_brez */
static void index2igra(int idx, int* tip, int* suit) {
    if (idx == 0) { *tip = ORC_NAPREJ; *suit = ORC_NO_KING; }
    else if (idx <= 12) { *tip = ORC_TRI + (idx - 1) / 4; *suit = (idx - 1) % 4; }
    else { static const int t[5] = { ORC_SOLO_TRI, ORC_SOLO_DVE, ORC_SOLO_ENA, ORC_BERAC, ORC_SOLO_BREZ };
           *tip = t[idx - 13]; *suit = ORC_NO_KING; }
}

typedef struct { uint64_t seed, gid; int tip[4]; uint32_t digit[16]; } bid_ctx;
static int want_uniform(void* p, int seat, int call) { (void)call; return ((bid_ctx*)p)->tip[seat]; }
static int want_bot(void* p, int seat, int call) {
    (void)seat;
    bid_ctx* b = (bid_ctx*)p;     /* np.random.choice([Naprej,Tri,Dve,Ena], p=[.5,1/6,1/6,1/6]), Igralec.py:151 */
    /* call i takes the i-th base-6 digit of words 0 and 1 of the bid block (eight batched draws each) */
    uint32_t u = call < 16 ? b->digit[call] : syn_draw(b->seed, b->gid, ST_BID, (uint32_t)(64 + call), 6);
    return u < 3 ? ORC_NAPREJ : (int)(ORC_TRI + (u - 3));
}

uint32_t syn_play_draw(uint64_t seed, uint64_t gid, uint32_t t, uint32_t n) {
    uint64_t pair = gid >> 1;
    uint32_t c[4] = { (uint32_t)pair, (uint32_t)(pair >> 32), ST_PLAY, t >> 2 };
    syn_philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    uint32_t lane = ((uint32_t)gid & 1u) * 4u + (t & 3u);
    uint32_t x = (c[lane >> 1] >> (16 * (lane & 1u))) & 0xFFFFu;
    uint32_t m = x * n, lo = m & 0xFFFFu;
    if (lo < n && lo < (65536u % n)) return syn_draw(seed, gid, ST_PLAY_RETRY, t, n);
    return m >> 16;
}

static int nth_lowest(uint64_t m, uint32_t r) {
    for (int c = 0; c < 54; c++) if ((m >> c) & 1) { if (r == 0) return c; r--; }
    return -1;
}

/* Talon exchange and uniform-random play-out of a game whose contract is set (orc_zacni_igro done): the declarer takes
   group 0 like Bot_igralec (Igralec.py:162), or a uniform group (word 3 of the setup block) when `random_group`, and lays
   k uniform discards (word 1 of the setup block); every card is a uniform legal one (syn_play_draw).  Returns 0, or -1 if
   the game is in an error state. */
static int syn_play_out(uint64_t seed, uint64_t gid, int random_group, orc_game* g, uint8_t cards[48],
                        uint8_t* group_out, uint64_t* discard_out) {
    *group_out = ORC_NO_GROUP; *discard_out = 0;
    memset(cards, 0xFF, 48);
    if (!g->error && g->phase == 1) {
        const int declarer = g->declarer;
        int k = orc_talon_k(g->contract);
        int grp = random_group ? (int)syn_draw(seed, gid, ST_FORCE, 3, g->group_cnt) : 0;
        /* discardable set after the pick-up: Roka.mozno_zalozit on hand + group (Igralec.py:163-166) */
        uint64_t avail = 0;
        orc_game tmp = *g;
        for (int j = 0; j < tmp.group_sz; j++) {
            int c = tmp.group[grp][j];
            int b = orc_iz_id(c).barva;
            tmp.hand[declarer][b][tmp.hand_n[declarer][b]++] = (uint8_t)c;
        }
        uint8_t mz[16];
        int nm = orc_mozno_zalozit(&tmp, declarer, mz);
        for (int i = 0; i < nm; i++) avail |= 1ull << mz[i];
        uint8_t d[3];
        uint64_t dm = 0;
        if (nm < k) { g->error = 1; return -1; }
        uint32_t nb[3], rd[3];                           /* word 1 of the setup block: the k discards, batched */
        for (int j = 0; j < k; j++) nb[j] = (uint32_t)(nm - j);
        syn_bdraws(seed, gid, ST_FORCE, ST_FORCE, 1, nb, k, rd);
        for (int j = 0; j < k; j++) {
            int c = nth_lowest(avail, rd[j]);
            d[j] = (uint8_t)c; avail &= ~(1ull << c); dm |= 1ull << c;
        }
        *group_out = (uint8_t)grp; *discard_out = dm;
        orc_menjaj(g, grp, d, k);
    }
    int t = 0;
    while (!g->error && g->phase == 2) {
        uint64_t m = orc_mozne_mask(g);
        uint32_t r = syn_play_draw(seed, gid, (uint32_t)t, (uint32_t)__builtin_popcountll(m));
        int c = nth_lowest(m, r);
        cards[t++] = (uint8_t)c;
        orc_igraj(g, c);
    }
    return g->error ? -1 : 0;
}

/* One whole deal with uniform-random players.  Returns 0, or -1 if the game hit an error state. */
int syn_rollout(uint64_t seed, uint64_t gid, int mode, orc_game* g, uint8_t perm[54],
                uint8_t cards[48], uint8_t* group_out, uint64_t* discard_out) {
    syn_deal(seed, gid, perm);
    orc_razdeli(g, perm);
    int contract, declarer = 0, king = ORC_NO_KING;
    if (mode == MODE_AUCTION_UNIFORM || mode == MODE_AUCTION_BOT) {
        bid_ctx b; b.seed = seed; b.gid = gid;
        int suit[4];
        if (mode == MODE_AUCTION_UNIFORM) {
            static const uint32_t n18[4] = { 18, 18, 18, 18 };
            uint32_t idx[4];
            syn_bdraws(seed, gid, ST_BID, ST_BID, 0, n18, 4, idx);
            for (int s = 0; s < 4; s++) index2igra((int)idx[s], &b.tip[s], &suit[s]);
        } else {
            static const uint32_t n6[8] = { 6, 6, 6, 6, 6, 6, 6, 6 };
            syn_bdraws(seed, gid, ST_BID, ST_BID, 0, n6, 8, b.digit);
            syn_bdraws(seed, gid, ST_BID, ST_BID, 1, n6, 8, b.digit + 8);
        }
        orc_licitacija(mode == MODE_AUCTION_UNIFORM ? want_uniform : want_bot, &b,
                       mode == MODE_AUCTION_UNIFORM, &declarer, &contract, 0);
        if (contract >= ORC_TRI && contract <= ORC_ENA)
            king = mode == MODE_AUCTION_UNIFORM ? suit[declarer] : (int)syn_draw(seed, gid, ST_FORCE, 2, 4);
    } else {
        static const uint32_t n344[3] = { 3, 4, 4 };      /* word 0 of the setup block: contract of the mix, declarer, king */
        uint32_t r[3];
        syn_bdraws(seed, gid, ST_FORCE, ST_FORCE, 0, n344, 3, r);
        contract = mode == MODE_NAVADNA_MIX ? (int)(ORC_TRI + r[0]) : mode;
        if (contract != ORC_KLOP) declarer = (int)r[1];
        if (contract >= ORC_TRI && contract <= ORC_ENA) king = (int)r[2];
    }
    orc_zacni_igro(g, contract, declarer, king);
    return syn_play_out(seed, gid, mode == MODE_AUCTION_UNIFORM, g, cards, group_out, discard_out);
}

/* An injected deal (perm, Igra.razdeli order) under a forced contract, played like the host-buffer entries of the CUDA
   path: talon group 0, discards and cards as in syn_rollout.  A row that is not a permutation of 0..53, or a declarer
   above 3, makes an error game (as does what orc_zacni_igro rejects: an unknown contract, a king game without a suit). */
static int syn_rollout_injected(uint64_t seed, uint64_t gid, const uint8_t perm[54], int contract, int declarer, int king,
                                orc_game* g, uint8_t cards[48], uint8_t* group_out, uint64_t* discard_out) {
    uint64_t seen = 0;
    for (int i = 0; i < 54; i++) if (perm[i] < 54) seen |= 1ull << perm[i];
    memset(g, 0, sizeof(*g));
    if (seen != (1ull << 54) - 1 || declarer > 3) {
        g->contract = contract; g->declarer = declarer; g->king = king;
        g->error = 1;
    } else {
        orc_razdeli(g, perm);
        orc_zacni_igro(g, contract, declarer, king);
    }
    return syn_play_out(seed, gid, 0, g, cards, group_out, discard_out);
}

/* Batch driver (OpenMP over games): synthetic deals and contracts of `mode`, or, with in_perm, the injected rows.  Any out
   pointer may be NULL.  out_hist counts the finished games by contract (the device's stats[8..17]). */
static void rollout_batch(uint64_t seed, uint64_t first_gid, int64_t n, int mode, const uint8_t* in_perm,
                          const uint8_t* in_contract, const uint8_t* in_declarer, const uint8_t* in_king,
                          int16_t* out_scores, uint8_t* out_plays, uint8_t* out_contract,
                          uint8_t* out_declarer, uint8_t* out_king, uint8_t* out_err,
                          uint8_t* out_perm, uint8_t* out_cards, uint8_t* out_group, uint64_t* out_discard,
                          int64_t* out_stats, int64_t* out_hist) {
    int64_t st[10] = { 0 }, hist[10] = { 0 };
#pragma omp parallel
    {
        int64_t loc[10] = { 0 }, lh[10] = { 0 };
#pragma omp for schedule(static)
        for (int64_t i = 0; i < n; i++) {
            orc_game g;
            uint8_t perm[54], cards[48], grp;
            uint64_t dm;
            uint64_t gid = first_gid + (uint64_t)i;
            if (in_perm) {
                memcpy(perm, in_perm + 54 * i, 54);
                syn_rollout_injected(seed, gid, perm, in_contract[i], in_declarer[i], in_king ? in_king[i] : ORC_NO_KING,
                                     &g, cards, &grp, &dm);
            } else {
                syn_rollout(seed, gid, mode, &g, perm, cards, &grp, &dm);
            }
            int fin = g.phase == 3 && !g.error;
            for (int s = 0; s < 4; s++) {
                int v = fin ? g.pisejo[s] : 0;
                if (out_scores) out_scores[4 * i + s] = (int16_t)v;
                loc[s] += v;
                loc[4 + ((s + gid) & 3)] += v;        /* seat s of game i is player (s+i)%4, Tarok.py:34 */
            }
            loc[8] += g.plays;
            loc[9] += g.error ? 1 : 0;
            if (fin && g.contract >= 0 && g.contract < 10) lh[g.contract]++;
            if (out_plays) out_plays[i] = (uint8_t)g.plays;
            if (out_contract) out_contract[i] = (uint8_t)g.contract;
            if (out_declarer) out_declarer[i] = (uint8_t)g.declarer;
            if (out_king) out_king[i] = (uint8_t)g.king;
            if (out_err) out_err[i] = (uint8_t)(g.error ? 1 : 0);
            if (out_perm) memcpy(out_perm + 54 * i, perm, 54);
            if (out_cards) memcpy(out_cards + 48 * i, cards, 48);
            if (out_group) out_group[i] = grp;
            if (out_discard) out_discard[i] = dm;
        }
#pragma omp critical
        for (int j = 0; j < 10; j++) { st[j] += loc[j]; hist[j] += lh[j]; }
    }
    if (out_stats) memcpy(out_stats, st, sizeof(st));
    if (out_hist) memcpy(out_hist, hist, sizeof(hist));
}

void syn_rollout_batch(uint64_t seed, uint64_t first_gid, int64_t n, int mode,
                       int16_t* out_scores, uint8_t* out_plays, uint8_t* out_contract,
                       uint8_t* out_declarer, uint8_t* out_king, uint8_t* out_err,
                       uint8_t* out_perm, uint8_t* out_cards, uint8_t* out_group, uint64_t* out_discard,
                       int64_t* out_stats /* [4 seat sums, 4 player sums, env steps, errors] */) {
    rollout_batch(seed, first_gid, n, mode, NULL, NULL, NULL, NULL, out_scores, out_plays, out_contract, out_declarer,
                  out_king, out_err, out_perm, out_cards, out_group, out_discard, out_stats, NULL);
}

/* n injected deals (perm [n,54]) under forced contracts (contract/declarer [n], king [n] or NULL = none), game i with id
   first_gid + i: what tarok_rollout_host / _records / _host_packed compute.  Same outputs as syn_rollout_batch (out_perm
   echoes the rows) plus the histogram of the finished games by contract. */
void syn_rollout_injected_batch(uint64_t seed, uint64_t first_gid, int64_t n, const uint8_t* perm, const uint8_t* contract,
                                const uint8_t* declarer, const uint8_t* king,
                                int16_t* out_scores, uint8_t* out_plays, uint8_t* out_contract,
                                uint8_t* out_declarer, uint8_t* out_king, uint8_t* out_err,
                                uint8_t* out_perm, uint8_t* out_cards, uint8_t* out_group, uint64_t* out_discard,
                                int64_t* out_stats, int64_t* out_hist) {
    rollout_batch(seed, first_gid, n, -1, perm, contract, declarer, king, out_scores, out_plays, out_contract, out_declarer,
                  out_king, out_err, out_perm, out_cards, out_group, out_discard, out_stats, out_hist);
}

void syn_deal_batch(uint64_t seed, uint64_t first_gid, int64_t n, uint8_t* out_perm) {
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < n; i++) syn_deal(seed, first_gid + (uint64_t)i, out_perm + 54 * i);
}

void syn_philox_kat(uint32_t c[4], uint32_t k0, uint32_t k1) { syn_philox4x32_10(c, k0, k1); }

/* thread control for the CPU-baseline legs (torchrun exports OMP_NUM_THREADS=1) */
#ifdef _OPENMP
#include <omp.h>
void syn_set_threads(int n) { if (n > 0) omp_set_num_threads(n); }
int syn_max_threads(void) { return omp_get_max_threads(); }
#else
void syn_set_threads(int n) { (void)n; }
int syn_max_threads(void) { return 1; }
#endif
