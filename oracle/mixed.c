/* TEST INFRASTRUCTURE ONLY -- the C oracle for mixed tables: Bot_igralec seats beside caller-driven (neural) seats.
 *
 * What tarok_auction_bots / tarok_exchange_bots / tarok_step_bots compute, restated on the oracle's list-based engine.  It
 * is compiled into its own library (libtarok_oracle_mixed.so, oracle/mixed.py) together with the two oracle sources it
 * builds on, which it includes whole so that it can use their internal helpers (the auction's bid filter, the batched
 * Philox draws, the Bot bidding digits) without changing them.
 */
#include "tarok_oracle.c"
#include "synth.c"

/* The same auction with the bidding semantics chosen per seat: bit s of `fresh_seats` set = seat s asks `want` afresh at
   every call (Bot_igralec, Igralec.py:151), otherwise it keeps its fixed intent (Nevronski_igralec, Igralec.py:295-304). */
static int bid_call_mixed(bidder* b, unsigned fresh_seats, int seat, int min_igra, int has_obv, int obv, int pred) {
    b->fixed = !((fresh_seats >> seat) & 1u);
    return bid_call(b, seat, min_igra, has_obv, obv, pred);
}

int orc_licitacija_mixed(orc_bid_fn want, void* ctx, unsigned fresh_seats, int* declarer, int* contract,
                         int* calls) {                        /* Igra.py:75-114 */
    bidder b;
    memset(&b, 0, sizeof(b));
    b.want = want; b.ctx = ctx;
    int lic = 0;
    int max_igra = ORC_TRI;
    for (int i = 1; i < 4; i++) {
        int nap = bid_call_mixed(&b, fresh_seats, i, max_igra, 0, 0, 0);
        if (nap != ORC_NAPREJ) lic |= 1 << i;
        if (nap > max_igra) max_igra = nap;
    }
    if (max_igra == ORC_TRI) {
        int nap = bid_call_mixed(&b, fresh_seats, 0, ORC_NAPREJ, 1, ORC_KLOP, 0);
        *declarer = 0; *contract = nap;
        if (calls) *calls = b.calls;
        return 0;
    } else {
        int nap = bid_call_mixed(&b, fresh_seats, 0, max_igra, 0, 0, 1);
        if (nap != ORC_NAPREJ) lic |= 1;
        if (nap > max_igra) max_igra = nap;
    }
    int ima_igro = 0;
    while (!((lic >> ima_igro) & 1)) ima_igro++;
    int guard = 0;
    while (__builtin_popcount((unsigned)lic) != 1) {
        int new_lic = 0;
        int keys[4], nk = 0;
        for (int k = 1; k < 4; k++) if ((lic >> k) & 1) keys[nk++] = k;
        if (lic & 1) keys[nk++] = 0;
        for (int j = 0; j < nk; j++) {
            int k = keys[j], nap;
            if (k == ima_igro) nap = bid_call_mixed(&b, fresh_seats, k, max_igra, 1, max_igra, 0);
            else nap = bid_call_mixed(&b, fresh_seats, k, max_igra, 0, 0, 0);
            if (nap != ORC_NAPREJ) { new_lic |= 1 << k; ima_igro = k; max_igra = nap; }
        }
        lic = new_lic;
        if (++guard > 64) return -1;
    }
    *declarer = ima_igro; *contract = max_igra;
    if (calls) *calls = b.calls;
    return 0;
}

/* ---- mixed tables: Bot_igralec seats beside caller-driven (neural) seats ------------------------------------------------
   What tarok_auction_bots / tarok_exchange_bots / tarok_step_bots compute for one game: bit s of `bots` = seat s is a Bot
   whose decisions are the Philox draws of the all-bot mode 18 (bids: the base-6 digits of the bid block by overall call
   number; king: setup-block word 2; exchange: group 0 and the discards of word 1; cards: syn_play_draw), the other seats
   bid their fixed index2igra intent (0..19: 18 Odprti_berac, 19 Klop; the king is the suit of the declarer's original
   intent), exchange neural_group / neural_discard and play cards[t]. */
static void index2igra20(int idx, int* tip, int* suit) {
    if (idx == 18) { *tip = ORC_ODPRTI_BERAC; *suit = ORC_NO_KING; }
    else if (idx == 19) { *tip = ORC_KLOP; *suit = ORC_NO_KING; }
    else index2igra(idx, tip, suit);
}

typedef struct { bid_ctx b; unsigned bots; } mixed_ctx;
static int want_mixed(void* p, int seat, int call) {
    mixed_ctx* m = (mixed_ctx*)p;
    return ((m->bots >> seat) & 1u) ? want_bot(&m->b, seat, call) : m->b.tip[seat];
}

/* Bot_igralec's exchange (Igralec.py:161-171) for a game waiting for one: group 0, k uniform discards (setup-block word 1). */
static int syn_bot_exchange(uint64_t seed, uint64_t gid, orc_game* g, uint8_t* group_out, uint64_t* discard_out) {
    const int declarer = g->declarer, k = orc_talon_k(g->contract);
    orc_game tmp = *g;
    for (int j = 0; j < tmp.group_sz; j++) {
        int c = tmp.group[0][j];
        int b = orc_iz_id(c).barva;
        tmp.hand[declarer][b][tmp.hand_n[declarer][b]++] = (uint8_t)c;
    }
    uint8_t mz[16], d[3];
    int nm = orc_mozno_zalozit(&tmp, declarer, mz);
    if (nm < k) { g->error = 1; return -1; }
    uint64_t avail = 0, dm = 0;
    for (int i = 0; i < nm; i++) avail |= 1ull << mz[i];
    uint32_t nb[3], rd[3];
    for (int j = 0; j < k; j++) nb[j] = (uint32_t)(nm - j);
    syn_bdraws(seed, gid, ST_FORCE, ST_FORCE, 1, nb, k, rd);
    for (int j = 0; j < k; j++) {
        int c = nth_lowest(avail, rd[j]);
        d[j] = (uint8_t)c; avail &= ~(1ull << c); dm |= 1ull << c;
    }
    *group_out = 0; *discard_out = dm;
    return orc_menjaj(g, 0, d, k);
}

/* Replays one mixed-table game: the auction, the king call, the exchange, and every play -- a bot's card is drawn here and
   checked against cards[t] (*mismatch = the first play where they differ, -1 none; the drawn card is the one played), a
   neural card must be legal (else the game becomes an error game).  cards may be NULL when every mover is a bot.  plays:
   the cards played (0xFF after the last).  A mask above 15, or an intent above 19 at a neural seat, is an error game.
   Returns 0, or -1 for an error game. */
int syn_replay_bots(uint64_t seed, uint64_t gid, const uint8_t perm[54], const uint8_t intents[4], uint8_t bots,
                    uint8_t neural_group, uint64_t neural_discard, const uint8_t* cards, orc_game* g, uint8_t plays[48],
                    uint8_t* group_out, uint64_t* discard_out, int* mismatch) {
    memset(g, 0, sizeof(*g));
    memset(plays, 0xFF, 48);
    *group_out = ORC_NO_GROUP; *discard_out = 0; *mismatch = -1;
    orc_razdeli(g, perm);
    mixed_ctx m;
    m.b.seed = seed; m.b.gid = gid; m.bots = bots & 15u;
    int suit[4], bad = bots > 15;
    for (int s = 0; s < 4; s++) {
        m.b.tip[s] = ORC_NAPREJ; suit[s] = ORC_NO_KING;
        if ((m.bots >> s) & 1u) continue;                     /* a bot seat's intent is never read */
        if (intents[s] > 19) bad = 1;
        else index2igra20(intents[s], &m.b.tip[s], &suit[s]);
    }
    if (m.bots) {                                             /* the sixteen base-6 digits of mode 18 */
        static const uint32_t n6[8] = { 6, 6, 6, 6, 6, 6, 6, 6 };
        syn_bdraws(seed, gid, ST_BID, ST_BID, 0, n6, 8, m.b.digit);
        syn_bdraws(seed, gid, ST_BID, ST_BID, 1, n6, 8, m.b.digit + 8);
    }
    int contract = ORC_NAPREJ, declarer = 0;
    if (!bad) orc_licitacija_mixed(want_mixed, &m, m.bots, &declarer, &contract, 0);
    if (bad) { g->contract = 15; g->error = 1; return -1; }
    int king = ORC_NO_KING;
    if (contract >= ORC_TRI && contract <= ORC_ENA)
        king = ((m.bots >> declarer) & 1u) ? (int)syn_draw(seed, gid, ST_FORCE, 2, 4) : suit[declarer];
    if (orc_zacni_igro(g, contract, declarer, king) != 0) return -1;
    if (g->phase == 1) {
        if ((m.bots >> g->declarer) & 1u) syn_bot_exchange(seed, gid, g, group_out, discard_out);
        else {
            menjaj_mask(g, neural_group, neural_discard);
            if (!g->error) { *group_out = neural_group; *discard_out = neural_discard; }
        }
    }
    for (int t = 0; !g->error && g->phase == 2; t++) {
        int c;
        if ((m.bots >> orc_na_potezi(g)) & 1u) {
            uint64_t mm = orc_mozne_mask(g);
            c = nth_lowest(mm, syn_play_draw(seed, gid, (uint32_t)t, (uint32_t)__builtin_popcountll(mm)));
            if (cards && cards[t] != c && *mismatch < 0) *mismatch = t;
        } else {
            c = cards ? cards[t] : 0xFF;
        }
        if (orc_igraj(g, c) == 0) plays[t] = (uint8_t)c;
    }
    return g->error ? -1 : 0;
}

/* Batch driver (OpenMP over games), game i = global game first_gid + i.  group / discard / cards may be NULL. */
void syn_replay_bots_batch(uint64_t seed, uint64_t first_gid, int64_t n, const uint8_t* perm, const uint8_t* intents,
                           const uint8_t* bots, const uint8_t* group, const uint64_t* discard, const uint8_t* cards,
                           uint8_t* out_contract, uint8_t* out_declarer, uint8_t* out_king, uint8_t* out_group,
                           uint64_t* out_discard, uint8_t* out_plays, int16_t* out_scores, uint8_t* out_err,
                           int8_t* out_mismatch) {
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < n; i++) {
        orc_game g;
        int mis;
        const int rc = syn_replay_bots(seed, first_gid + (uint64_t)i, perm + 54 * i, intents + 4 * i, bots[i],
                                       group ? group[i] : ORC_NO_GROUP, discard ? discard[i] : 0, cards ? cards + 48 * i : NULL,
                                       &g, out_plays + 48 * i, out_group + i, out_discard + i, &mis);
        const int fin = rc == 0 && g.phase == 3;
        for (int s = 0; s < 4; s++) out_scores[4 * i + s] = fin ? g.pisejo[s] : 0;
        out_contract[i] = (uint8_t)g.contract; out_declarer[i] = (uint8_t)g.declarer; out_king[i] = (uint8_t)g.king;
        out_err[i] = (uint8_t)(rc != 0); out_mismatch[i] = (int8_t)mis;
    }
}
