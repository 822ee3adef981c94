/* TEST INFRASTRUCTURE ONLY -- see tarok_oracle.h.  Plain-C restatement of the reference rules. */
#include "tarok_oracle.h"

#include <math.h>
#include <string.h>

/* ------------------------------------------------------------------ Karta.py */

int orc_v_id(int barva, int st) {                 /* Karta.py:19-23 */
    if (barva == ORC_TAROK) return 4 * 8 + st - 1;
    return barva * 8 + st - 1;
}

orc_karta orc_iz_id(int id) {                     /* Karta.py:31-47 */
    orc_karta k;
    if (id > 31) { k.barva = ORC_TAROK; k.st = (uint8_t)(id - 31); }
    else { k.barva = (uint8_t)(id / 8); k.st = (uint8_t)(id % 8 + 1); }
    return k;
}

int orc_vrednost(int id) {                        /* Karta.py:10-16 */
    orc_karta k = orc_iz_id(id);
    if (k.barva == ORC_TAROK && (k.st == 1 || k.st == 21 || k.st == 22)) return 5;
    else if (k.st > 4) return k.st - 3;           /* also taroks V.. : the bug is part of the contract */
    else return 1;
}

static int karta_lt(int a, int b) {               /* Karta.__lt__, Karta.py:61-66 */
    orc_karta x = orc_iz_id(a), y = orc_iz_id(b);
    if (x.barva != y.barva) return x.barva < y.barva;
    return x.st < y.st;
}

/* ------------------------------------------------------------------ Roka.py */

int orc_vrednost_stiha(const uint8_t* ids, int n) {   /* Roka.py:72-95 */
    int vrednost = 0;
    for (int i = 0; i < n; i++) {
        orc_karta k = orc_iz_id(ids[i]);
        if (k.barva == ORC_TAROK) {
            if (1 < k.st && k.st < 21) vrednost += 1;
            else vrednost += 5;
        } else {
            if (4 < k.st) vrednost += k.st - 3;
            else vrednost += 1;
        }
    }
    if (n == 1 || n == 2) return vrednost - 1;
    return vrednost - 2;
}

int orc_prestej(const uint8_t* ids, int n) {          /* tri_po_tri Roka.py:55-59 + prestej :96-98 */
    int s = 0;
    for (int i = 0; i < n / 3; i++) s += orc_vrednost_stiha(ids + 3 * i, 3);
    if (n % 3 != 0) s += orc_vrednost_stiha(ids + n - (n % 3), n % 3);
    return s;
}

static void roka_remove(orc_game* g, int seat, int card) {   /* Roka.igraj_karto, Roka.py:15-16 */
    int b = orc_iz_id(card).barva;
    uint8_t* l = g->hand[seat][b];
    int n = g->hand_n[seat][b];
    for (int i = 0; i < n; i++)
        if (l[i] == card) {
            memmove(l + i, l + i + 1, (size_t)(n - i - 1));
            g->hand_n[seat][b] = (uint8_t)(n - 1);
            return;
        }
}

static void roka_append(orc_game* g, int seat, int card) {   /* Roka.dodaj_karte, Roka.py:18-21 */
    int b = orc_iz_id(card).barva;
    g->hand[seat][b][g->hand_n[seat][b]++] = (uint8_t)card;
}

static int roka_contains(const orc_game* g, int seat, int card) {   /* Roka.__contains__ */
    int b = orc_iz_id(card).barva;
    for (int i = 0; i < g->hand_n[seat][b]; i++)
        if (g->hand[seat][b][i] == card) return 1;
    return 0;
}

int orc_mozno_zalozit(const orc_game* g, int seat, uint8_t* out) {   /* Roka.py:23-27 */
    int n = 0;
    for (int b = 0; b < 5; b++)
        for (int i = 0; i < g->hand_n[seat][b]; i++)
            if (orc_vrednost(g->hand[seat][b][i]) < 5) out[n++] = g->hand[seat][b][i];
    return n;
}

/* ------------------------------------------------------------------ Igra.py */

void orc_razdeli(orc_game* g, const uint8_t perm[54]) {   /* Igra.py:65-73 + Roka.__init__ */
    memset(g, 0, sizeof(*g));
    for (int s = 0; s < 4; s++) {
        for (int i = 0; i < 12; i++) roka_append(g, s, perm[12 * s + i]);
        for (int b = 0; b < 5; b++) {                      /* v.sort() per suit, Roka.py:10-11 */
            uint8_t* l = g->hand[s][b];
            int n = g->hand_n[s][b];
            for (int i = 1; i < n; i++) {
                uint8_t x = l[i];
                int j = i - 1;
                while (j >= 0 && karta_lt(x, l[j])) { l[j + 1] = l[j]; j--; }
                l[j + 1] = x;
            }
        }
    }
    for (int i = 0; i < 6; i++) g->talon[i] = perm[48 + i];
    g->talon_n = 6;
    g->contract = ORC_NAPREJ;
    g->king = ORC_NO_KING;
    g->chosen_group = ORC_NO_GROUP;
    g->last_winner = -1;
    g->phase = 0;
}

/* Igralec.licitiram filter, Igralec.py:58-74 */
static int licitiram_filter(int want, int min_igra, int has_obv, int obvezno, int prednost) {
    if (prednost) {
        if (want >= min_igra) return want;
        return has_obv ? obvezno : ORC_NAPREJ;
    } else {
        if (want > min_igra) return want;
        return has_obv ? obvezno : ORC_NAPREJ;
    }
}

typedef struct {
    orc_bid_fn want; void* ctx; int fixed; int intent[4]; int have[4]; int calls;
} bidder;

static int bid_call(bidder* b, int seat, int min_igra, int has_obv, int obv, int pred) {
    int w;
    if (b->fixed) {
        if (!b->have[seat]) { b->intent[seat] = b->want(b->ctx, seat, b->calls); b->have[seat] = 1; }
        w = b->intent[seat];
    } else {
        w = b->want(b->ctx, seat, b->calls);
    }
    b->calls++;
    int r = licitiram_filter(w, min_igra, has_obv, obv, pred);
    if (b->fixed) b->intent[seat] = r;      /* Nevronski_igralec.licitiram, Igralec.py:304 */
    return r;
}

int orc_licitacija(orc_bid_fn want, void* ctx, int fixed_intent, int* declarer, int* contract,
                   int* calls) {                              /* Igra.py:75-114 */
    bidder b;
    memset(&b, 0, sizeof(b));
    b.want = want; b.ctx = ctx; b.fixed = fixed_intent;
    int lic = 0;                       /* set of seats as bitmask */
    int max_igra = ORC_TRI;
    for (int i = 1; i < 4; i++) {
        int nap = bid_call(&b, i, max_igra, 0, 0, 0);
        if (nap != ORC_NAPREJ) lic |= 1 << i;
        if (nap > max_igra) max_igra = nap;
    }
    if (max_igra == ORC_TRI) {
        int nap = bid_call(&b, 0, ORC_NAPREJ, 1, ORC_KLOP, 0);
        *declarer = 0; *contract = nap;
        if (calls) *calls = b.calls;
        return 0;
    } else {
        int nap = bid_call(&b, 0, max_igra, 0, 0, 1);
        if (nap != ORC_NAPREJ) lic |= 1;
        if (nap > max_igra) max_igra = nap;
    }
    int ima_igro = 0;
    while (!((lic >> ima_igro) & 1)) ima_igro++;             /* min(lic) */
    int guard = 0;
    while (__builtin_popcount((unsigned)lic) != 1) {
        int new_lic = 0;
        int keys[4], nk = 0;
        for (int k = 1; k < 4; k++) if ((lic >> k) & 1) keys[nk++] = k;
        if (lic & 1) keys[nk++] = 0;                          /* keys[1:]+[0] */
        for (int j = 0; j < nk; j++) {
            int k = keys[j], nap;
            if (k == ima_igro) nap = bid_call(&b, k, max_igra, 1, max_igra, 0);
            else nap = bid_call(&b, k, max_igra, 0, 0, 0);
            if (nap != ORC_NAPREJ) { new_lic |= 1 << k; ima_igro = k; max_igra = nap; }
        }
        lic = new_lic;
        if (++guard > 64) return -1;
    }
    *declarer = ima_igro; *contract = max_igra;
    if (calls) *calls = b.calls;
    return 0;
}

int orc_talon_k(int contract) {                               /* Navadna_igra.py:36-58 */
    switch (contract) {
        case ORC_TRI: case ORC_SOLO_TRI: return 3;
        case ORC_DVE: case ORC_SOLO_DVE: return 2;
        case ORC_ENA: case ORC_SOLO_ENA: return 1;
        default: return 0;
    }
}

static int is_navadna(int c) { return (c >= ORC_TRI && c <= ORC_SOLO_ENA) || c == ORC_SOLO_BREZ; }
static int is_king_game(int c) { return c >= ORC_TRI && c <= ORC_ENA; }
static int is_berac(int c) { return c == ORC_BERAC || c == ORC_ODPRTI_BERAC; }

int orc_zacni_igro(orc_game* g, int contract, int declarer, int king) {   /* Igra.py:38-53 */
    g->contract = contract; g->declarer = declarer;
    g->king = is_king_game(contract) ? king : ORC_NO_KING;   /* king only asked for Ena/Dve/Tri, Igra.py:42-43 */
    memset(g->ekipa, 0, sizeof(g->ekipa));
    if (declarer < 0 || declarer > 3) { g->error = 1; return -1; }   /* no such player, whatever the contract (Klop too) */
    if (is_navadna(contract)) {
        if (is_king_game(contract)) {                         /* Navadna_igra.py:20-25 */
            if (king < 0 || king > 3) { g->error = 1; return -1; }   /* assert barva_kralja != TAROK */
            int kralj = orc_v_id(king, 8);
            for (int s = 0; s < 4; s++)
                g->ekipa[s] = (uint8_t)(roka_contains(g, s, kralj) || s == declarer);
        } else {
            g->ekipa[declarer] = 1;                           /* Navadna_igra.py:26-30 */
        }
        int korak = orc_talon_k(contract);                    /* odpri_talon, Navadna_igra.py:36-44 */
        if (korak == 0) korak = 1;                            /* Solo_brez falls in the else branch */
        g->group_sz = (uint8_t)korak;
        g->group_cnt = (uint8_t)(6 / korak);
        for (int i = 0; i < g->group_cnt; i++) {
            g->group_alive[i] = 1;
            for (int j = 0; j < korak; j++) g->group[i][j] = g->talon[i * korak + j];
        }
        g->zacne = 0;                                          /* Navadna_igra.py:70 */
        g->phase = (contract == ORC_SOLO_BREZ) ? 2 : 1;
    } else if (contract == ORC_KLOP) {
        g->declarer = 0;
        g->zacne = 0;                                          /* Klop.py:26 */
        g->phase = 2;
    } else if (is_berac(contract)) {
        g->zacne = declarer;                                   /* Berac.py:15 */
        g->phase = 2;
    } else {
        g->error = 1;                                          /* "Igra ni definirana", Igra.py:55 */
        return -1;
    }
    return 0;
}

int orc_menjaj(orc_game* g, int group, const uint8_t* discards, int k) {
    /* Navadna_igra.py:59-66 (engine side) + Bot_igralec.menjaj_iz_talona Igralec.py:161-171 (player side) */
    if (g->phase != 1 || k != orc_talon_k(g->contract) || group < 0 || group >= g->group_cnt) {
        g->error = 1; return -1;
    }
    int d = g->declarer;
    orc_game t = *g;                                           /* a refused exchange leaves the game as it was */
    for (int j = 0; j < t.group_sz; j++) roka_append(&t, d, t.group[group][j]);
    uint8_t mozno[16];
    int nm = orc_mozno_zalozit(&t, d, mozno);
    if (nm < k) { g->error = 1; return -1; }                   /* random.sample would raise (Q19) */
    for (int i = 0; i < k; i++) {
        int ok = 0;
        for (int j = 0; j < nm; j++) if (mozno[j] == discards[i]) ok = 1;
        for (int j = 0; j < i; j++) if (discards[j] == discards[i]) ok = 0;
        if (!ok) { g->error = 1; return -1; }
    }
    for (int i = 0; i < k; i++) {
        t.pile[d][t.pile_n[d]++] = discards[i];                /* kupcek.extend(izberi) */
        roka_remove(&t, d, discards[i]);
    }
    t.chosen_group = (uint8_t)group;
    t.group_alive[group] = 0;                                  /* del kupcki_talona[stevilka_kupcka] */
    t.phase = 2;
    *g = t;
    return 0;
}

/* ------------------------------------------------------------------ play */

static int primerjaj_karti(int k1, int k2) {   /* Navadna_igra.py:150-156 == Klop.py:88-94 */
    orc_karta a = orc_iz_id(k1), b = orc_iz_id(k2);
    if (a.barva == b.barva) return a.st < b.st;
    else if (b.barva == ORC_TAROK) return 1;
    else return 0;
}

static int pobere_stih(const uint8_t* stih) {  /* Navadna_igra.py:143-148 == Klop.py:81-86 */
    int zmaga = 0;
    for (int i = 1; i < 4; i++)
        if (primerjaj_karti(stih[zmaga], stih[i])) zmaga = i;
    return zmaga;
}

static int vse_sorted(const orc_game* g, int seat, uint8_t* out) {   /* vse.extend(...); vse.sort() */
    int n = 0;
    for (int b = 0; b < 5; b++)
        for (int i = 0; i < g->hand_n[seat][b]; i++) out[n++] = g->hand[seat][b][i];
    for (int i = 1; i < n; i++) {
        uint8_t x = out[i];
        int j = i - 1;
        while (j >= 0 && karta_lt(x, out[j])) { out[j + 1] = out[j]; j--; }
        out[j + 1] = x;
    }
    return n;
}

static int is_palcka(int id) { orc_karta k = orc_iz_id(id); return k.barva == ORC_TAROK && k.st == 1; }

static int mozne_navadna(const orc_game* g, int seat, int spodnja, uint8_t* out) {
    /* Navadna_igra.py:158-168 */
    if (spodnja >= 0) {
        int b = orc_iz_id(spodnja).barva;
        if (g->hand_n[seat][b] > 0) {
            memcpy(out, g->hand[seat][b], g->hand_n[seat][b]);
            return g->hand_n[seat][b];
        } else if (g->hand_n[seat][ORC_TAROK] > 0) {
            memcpy(out, g->hand[seat][ORC_TAROK], g->hand_n[seat][ORC_TAROK]);
            return g->hand_n[seat][ORC_TAROK];
        }
    }
    return vse_sorted(g, seat, out);
}

static int mozne_klop(const orc_game* g, int seat, int spodnja, uint8_t* out) {
    /* Klop.py:96-133, literal -- including the filter that is computed and then not used (:104) */
    if (spodnja >= 0 && g->hand_n[seat][orc_iz_id(spodnja).barva] > 0) {
        const uint8_t* mozne = g->hand[seat][orc_iz_id(spodnja).barva];
        int nm = g->hand_n[seat][orc_iz_id(spodnja).barva];
        int n_filtrirano = 0;
        uint8_t filtrirano[16];
        for (int i = 0; i < nm; i++)
            if (primerjaj_karti(spodnja, mozne[i])) filtrirano[n_filtrirano++] = mozne[i];
        if (n_filtrirano > 0) {
            uint8_t brez_palcke[16];
            int nb = 0;
            for (int i = 0; i < nm; i++) if (!is_palcka(mozne[i])) brez_palcke[nb++] = mozne[i];
            if (nb > 0) { memcpy(out, brez_palcke, (size_t)nb); return nb; }
            memcpy(out, filtrirano, (size_t)n_filtrirano);
            return n_filtrirano;
        } else {
            int n = 0;
            if (nm > 1) { for (int i = 0; i < nm; i++) if (!is_palcka(mozne[i])) out[n++] = mozne[i]; }
            else { memcpy(out, mozne, (size_t)nm); n = nm; }
            return n;
        }
    } else if (spodnja >= 0 && g->hand_n[seat][ORC_TAROK] > 0) {
        const uint8_t* taroki = g->hand[seat][ORC_TAROK];
        int nt = g->hand_n[seat][ORC_TAROK];
        int n_filtrirano = 0;
        for (int i = 0; i < nt; i++) if (primerjaj_karti(spodnja, taroki[i])) n_filtrirano++;
        if (n_filtrirano > 0) {
            int n = 0;
            for (int i = 0; i < nt; i++) if (orc_iz_id(taroki[i]).st != 1) out[n++] = taroki[i];
            if (n == 0) { memcpy(out, taroki, (size_t)nt); n = nt; }
            return n;
        }
        memcpy(out, taroki, (size_t)nt);
        return nt;
    } else {
        uint8_t vse[16];
        int n = vse_sorted(g, seat, vse);
        if (n > 1) {
            int m = 0;
            for (int i = 0; i < n; i++) if (!is_palcka(vse[i])) out[m++] = vse[i];
            return m;
        }
        memcpy(out, vse, (size_t)n);
        return n;
    }
}

int orc_na_potezi(const orc_game* g) { return (g->zacne + g->pos) % 4; }

int orc_mozne_karte(const orc_game* g, uint8_t* out) {
    int seat = orc_na_potezi(g);
    int spodnja = g->pos > 0 ? g->stih[0] : -1;
    if (is_navadna(g->contract)) return mozne_navadna(g, seat, spodnja, out);
    return mozne_klop(g, seat, spodnja, out);                 /* Berac inherits, Berac.py:4 */
}

uint64_t orc_mozne_mask(const orc_game* g) {
    uint8_t m[16];
    int n = orc_mozne_karte(g, m);
    uint64_t r = 0;
    for (int i = 0; i < n; i++) r |= 1ull << m[i];
    return r;
}

static void konec_navadna(orc_game* g) {                       /* Navadna_igra.py:80-113 */
    uint8_t skupek[64], skupek2[64];
    int n1 = 0, n2 = 0, st_ekipa = 0;
    for (int s = 0; s < 4; s++) {
        if (g->ekipa[s]) { memcpy(skupek + n1, g->pile[s], g->pile_n[s]); n1 += g->pile_n[s]; st_ekipa++; }
    }
    for (int s = 0; s < 4; s++) {
        if (!g->ekipa[s]) { memcpy(skupek2 + n2, g->pile[s], g->pile_n[s]); n2 += g->pile_n[s]; }
    }
    int king_in_pile = 0;
    if (g->king != ORC_NO_KING) {
        int kralj = orc_v_id(g->king, 8);
        for (int i = 0; i < g->pile_n[g->declarer]; i++) if (g->pile[g->declarer][i] == kralj) king_in_pile = 1;
    }
    int to_team = g->contract != ORC_SOLO_BREZ && st_ekipa == 1 && g->king != ORC_NO_KING && king_in_pile;
    for (int i = 0; i < g->group_cnt; i++) {
        if (!g->group_alive[i]) continue;
        for (int j = 0; j < g->group_sz; j++) {
            if (to_team) skupek[n1++] = g->group[i][j];
            else skupek2[n2++] = g->group[i][j];
        }
    }
    int vrednost = orc_prestej(skupek, n1);
    int razlika = vrednost - 35;
    razlika = (int)nearbyint((double)razlika / 5.0) * 5;       /* int(round(razlika/5))*5, half-even */
    int igra = g->contract * 10;
    for (int s = 0; s < 4; s++) {
        if (g->ekipa[s]) g->pisejo[s] = (int16_t)(vrednost > 35 ? igra + razlika : -igra + razlika);
        else g->pisejo[s] = 0;
    }
}

static void konec_klop(orc_game* g) {                          /* Klop.py:36-42 */
    int any = 0;
    for (int s = 0; s < 4; s++) {
        g->pisejo[s] = (int16_t)(-orc_prestej(g->pile[s], g->pile_n[s]));
        if (g->pisejo[s] < -35) any = 1;
    }
    if (any) {
        for (int s = 0; s < 4; s++) {
            if (orc_prestej(g->pile[s], g->pile_n[s]) < -35) g->pisejo[s] = -70;   /* never true */
            else g->pisejo[s] = 0;
        }
    }
}

int orc_igraj(orc_game* g, int card) {
    if (g->phase != 2 || g->error) { g->error = 1; return -1; }
    int seat = orc_na_potezi(g);
    uint8_t mozne[16];
    int nm = orc_mozne_karte(g, mozne), ok = 0;
    for (int i = 0; i < nm; i++) if (mozne[i] == card) ok = 1;
    if (!ok) { g->error = 1; return -1; }                      /* 'Karte ne mores igarti' */
    roka_remove(g, seat, card);                                /* Igralec.igraj_karto, Igralec.py:82-85 */
    g->hist[g->plays++] = (uint8_t)((seat << 6) | card);
    g->stih[g->stih_n++] = (uint8_t)card;
    g->pos++;
    if (g->pos < 4) return 0;
    /* end of krog */
    if (g->contract == ORC_KLOP && g->talon_n > 0)             /* Klop.py:67-71 (Berac: add_talon=False) */
        g->stih[g->stih_n++] = g->talon[--g->talon_n];
    int zmaga = pobere_stih(g->stih);
    int w = (g->zacne + zmaga) % 4;
    memcpy(g->pile[w] + g->pile_n[w], g->stih, (size_t)g->stih_n);
    g->pile_n[w] = (uint8_t)(g->pile_n[w] + g->stih_n);
    g->last_winner = w;
    g->zacne = w;
    g->pos = 0; g->stih_n = 0;
    g->tricks++;
    if (is_berac(g->contract)) {                               /* Berac.py:29-40 */
        int v = g->contract == ORC_ODPRTI_BERAC ? 90 : 70;
        if (w == g->declarer) {
            memset(g->pisejo, 0, sizeof(g->pisejo));
            g->pisejo[g->declarer] = (int16_t)(-v);
            g->phase = 3;
        } else if (g->tricks == 12) {
            memset(g->pisejo, 0, sizeof(g->pisejo));
            g->pisejo[g->declarer] = (int16_t)v;
            g->phase = 3;
        }
    } else if (g->tricks == 12) {
        if (g->contract == ORC_KLOP) konec_klop(g);
        else konec_navadna(g);
        g->phase = 3;
    }
    return 0;
}

/* ------------------------------------------------------------------ batch drivers */

static uint64_t hand_mask(const orc_game* g, int s) {
    uint64_t m = 0;
    for (int b = 0; b < 5; b++) for (int i = 0; i < g->hand_n[s][b]; i++) m |= 1ull << g->hand[s][b][i];
    return m;
}
static uint64_t pile_mask(const orc_game* g, int s) {
    uint64_t m = 0;
    for (int i = 0; i < g->pile_n[s]; i++) m |= 1ull << g->pile[s][i];
    return m;
}
static uint64_t talon_mask(const orc_game* g) {
    uint64_t m = 0;
    if (is_navadna(g->contract) && g->group_cnt) {             /* (a rejected contract never split the talon) */
        for (int i = 0; i < g->group_cnt; i++)
            if (g->group_alive[i]) for (int j = 0; j < g->group_sz; j++) m |= 1ull << g->group[i][j];
    } else {
        for (int i = 0; i < g->talon_n; i++) m |= 1ull << g->talon[i];
    }
    return m;
}

/* Deal + contract of one game of the batch drivers.  A row that is not a permutation of 0..53 is an error game with
   nothing dealt, the rule k_set_deals applies; orc_razdeli would index past its lists. */
static void deal_and_start(orc_game* g, const uint8_t perm[54], int contract, int declarer, int king) {
    uint64_t seen = 0;
    for (int i = 0; i < 54; i++) if (perm[i] < 54) seen |= 1ull << perm[i];
    if (seen != (1ull << 54) - 1) {
        memset(g, 0, sizeof(*g));
        g->error = 1;
        return;
    }
    orc_razdeli(g, perm);
    orc_zacni_igro(g, contract, declarer, king);
}

/* The exchange as a discard bitboard: a mask with more than three cards or a bit above card 53 is an invalid exchange. */
static void menjaj_mask(orc_game* g, int group, uint64_t mask) {
    uint8_t d[3] = { 0, 0, 0 };
    int k = 0;
    for (int c = 0; c < 54 && k < 3; c++) if ((mask >> c) & 1) d[k++] = (uint8_t)c;
    int kk = __builtin_popcountll(mask);
    orc_menjaj(g, group, d, (kk > 3 || (mask >> 54)) ? 99 : kk);
}

void orc_replay_batch(int64_t n, const uint8_t* perm, const uint8_t* contract, const uint8_t* declarer,
                      const uint8_t* king, const uint8_t* group, const uint64_t* discard_mask,
                      const uint8_t* cards, uint8_t* out_seat, uint64_t* out_mask, uint8_t* out_winner,
                      int16_t* out_scores, uint8_t* out_plays, uint8_t* out_err,
                      uint64_t* out_hands, uint64_t* out_piles, uint64_t* out_talon) {
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < n; i++) {
        orc_game g;
        deal_and_start(&g, perm + 54 * i, contract[i], declarer[i], king[i]);
        if (!g.error && g.phase == 1) menjaj_mask(&g, group[i], discard_mask[i]);
        for (int t = 0; t < 48; t++) { if (out_seat) out_seat[48 * i + t] = 0xFF; if (out_mask) out_mask[48 * i + t] = 0; }
        for (int t = 0; t < 12; t++) if (out_winner) out_winner[12 * i + t] = 0xFF;
        int t = 0;
        while (!g.error && g.phase == 2 && t < 48) {
            int c = cards[48 * i + t];
            if (c == 0xFF) break;
            if (out_seat) out_seat[48 * i + t] = (uint8_t)orc_na_potezi(&g);
            if (out_mask) out_mask[48 * i + t] = orc_mozne_mask(&g);
            int tr = g.tricks;
            orc_igraj(&g, c);
            if (!g.error && g.tricks != tr && out_winner) out_winner[12 * i + tr] = (uint8_t)g.last_winner;
            if (!g.error) t++;
        }
        if (out_plays) out_plays[i] = (uint8_t)g.plays;
        if (out_err) out_err[i] = (uint8_t)(g.error ? 1 : 0);
        for (int s = 0; s < 4; s++) {
            if (out_scores) out_scores[4 * i + s] = g.phase == 3 ? g.pisejo[s] : 0;
            if (out_hands) out_hands[4 * i + s] = hand_mask(&g, s);
            if (out_piles) out_piles[4 * i + s] = pile_mask(&g, s);
        }
        if (out_talon) out_talon[i] = talon_mask(&g);
    }
}

/* The ordered lists the neural player decides over, with the same teacher forcing as orc_replay_batch:
   per play (and for the first 0xFF of a game still being played: the decision pending there) the `mozne` list in the reference's order (Navadna_igra.py:158-168 / Klop.py:96-133) and the seat to move;
   per trick the value the replay target uses (Roka.vrednost_stiha of the trick incl. Klop's talon card, Roka.py:72-95);
   per exchange the `mozno_zalozit()` list after the pick-up (Roka.py:23-27, Igralec.py:376-380) and the talon groups
   (Navadna_igra.py:36-44).  Unused slots are 0xFF; values of unplayed tricks are 0. */
void orc_lists_batch(int64_t n, const uint8_t* perm, const uint8_t* contract, const uint8_t* declarer,
                     const uint8_t* king, const uint8_t* group, const uint64_t* discard_mask, const uint8_t* cards,
                     uint8_t* out_mozne, uint8_t* out_mozne_n, uint8_t* out_seat, int16_t* out_trick_value,
                     uint8_t* out_zalozit, uint8_t* out_zalozit_n, uint8_t* out_groups) {
#pragma omp parallel for schedule(static)
    for (int64_t i = 0; i < n; i++) {
        orc_game g;
        deal_and_start(&g, perm + 54 * i, contract[i], declarer[i], king[i]);
        memset(out_mozne + 48 * 16 * i, 0xFF, 48 * 16);
        memset(out_mozne_n + 48 * i, 0, 48);
        memset(out_seat + 48 * i, 0xFF, 48);
        for (int k = 0; k < 12; k++) out_trick_value[12 * i + k] = 0;
        memset(out_zalozit + 16 * i, 0xFF, 16);
        out_zalozit_n[i] = 0;
        memset(out_groups + 18 * i, 0xFF, 18);
        if (!g.error && g.phase == 1) {
            for (int a = 0; a < g.group_cnt; a++)
                for (int j = 0; j < g.group_sz; j++) out_groups[18 * i + 3 * a + j] = g.group[a][j];
            if (group[i] < g.group_cnt) {
                orc_game tmp = g;
                for (int j = 0; j < tmp.group_sz; j++) roka_append(&tmp, tmp.declarer, tmp.group[group[i]][j]);
                out_zalozit_n[i] = (uint8_t)orc_mozno_zalozit(&tmp, tmp.declarer, out_zalozit + 16 * i);
            }
            menjaj_mask(&g, group[i], discard_mask[i]);
        }
        int t = 0;
        while (!g.error && g.phase == 2 && t < 48) {
            int c = cards[48 * i + t];
            out_seat[48 * i + t] = (uint8_t)orc_na_potezi(&g);
            out_mozne_n[48 * i + t] = (uint8_t)orc_mozne_karte(&g, out_mozne + (48 * i + t) * 16);
            if (c == 0xFF) break;                                  /* the pending decision is written too */
            int tr = g.tricks, before[4];
            for (int s = 0; s < 4; s++) before[s] = g.pile_n[s];
            orc_igraj(&g, c);
            if (g.error) break;
            if (g.tricks != tr) {
                int w = g.last_winner;
                out_trick_value[12 * i + tr] = (int16_t)orc_vrednost_stiha(g.pile[w] + before[w], g.pile_n[w] - before[w]);
            }
            t++;
        }
    }
}

typedef struct { const int8_t* v; } arr_ctx;
static int want_fixed(void* ctx, int seat, int call) { (void)call; return ((arr_ctx*)ctx)->v[seat]; }
static int want_scripted(void* ctx, int seat, int call) { (void)seat; return call < 16 ? ((arr_ctx*)ctx)->v[call] : ORC_NAPREJ; }

void orc_auction_fixed_batch(int64_t n, const int8_t* intents, uint8_t* declarer, uint8_t* contract,
                             uint8_t* calls) {
    for (int64_t i = 0; i < n; i++) {
        arr_ctx c = { intents + 4 * i };
        int d = 0, k = 0, nc = 0;
        orc_licitacija(want_fixed, &c, 1, &d, &k, &nc);
        declarer[i] = (uint8_t)d; contract[i] = (uint8_t)k; if (calls) calls[i] = (uint8_t)nc;
    }
}

void orc_auction_scripted_batch(int64_t n, const int8_t* draws, uint8_t* declarer, uint8_t* contract,
                                uint8_t* calls) {
    for (int64_t i = 0; i < n; i++) {
        arr_ctx c = { draws + 16 * i };
        int d = 0, k = 0, nc = 0;
        orc_licitacija(want_scripted, &c, 0, &d, &k, &nc);
        declarer[i] = (uint8_t)d; contract[i] = (uint8_t)k; if (calls) calls[i] = (uint8_t)nc;
    }
}

void orc_prestej_batch(int64_t n, const uint8_t* ids, const uint8_t* len, int stride, int32_t* out) {
    for (int64_t i = 0; i < n; i++) out[i] = orc_prestej(ids + (int64_t)stride * i, len[i]);
}
