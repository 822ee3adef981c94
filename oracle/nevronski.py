"""TEST INFRASTRUCTURE ONLY -- a plain numpy / float64 restatement of the reference's neural player.

What ``Nevronski_igralec`` computes for a decision, vectorised over games (SURVEY.md A.4; the header comments of
``tarok_b200/csrc/tarok_obs.cuh`` state the same definitions):

* ``observation``  -- ``stanje_v_vektor_rek_navadna`` (Igralec.py:453-533) of the seat that makes card play t;
* ``choose_card``  -- ``igraj_karto`` (Igralec.py:344-355): ``np.argmax(q[mozne])`` in the order of the list ``mozne``;
* ``choose_exchange`` -- ``menjaj_iz_talona`` (Igralec.py:365-385);
* ``targets``      -- ``rezultat_stiha`` / ``rezultat_igre`` (Igralec.py:387-446), in float64.

It is written from those definitions and not from the kernels.  The ordered lists the player decides over (``mozne``,
``mozno_zalozit()``, the talon groups) and the trick values come from the C oracle (``oracle.lists``), whose data model
is the reference's own.  Exploration follows the device's Philox definition (DESIGN.md section 4), the only place where
the reference's ``random.random()`` has no fixed value to compare with.  ``tarok_b200`` never imports this file.

Games are given as a dict of numpy arrays: perm [n,54], contract, declarer, king, group [n], discard_mask uint64 [n],
cards uint8 [n,48] (0xFF = no play).
"""
from __future__ import annotations

import numpy as np

from . import oracle as O

NO_PLAY = 0xFF
ST_EXPLORE = 8                      # Philox stream of the neural player's exploration draws
U1 = np.uint64(1)


def net_type(contract):
    """Nevronski_igralec.tip_igre_v_tip_izbire (Igralec.py:179-188): 0 Klop, 1 Navadna_igra, 2 Solo, 3 Berac."""
    c = np.asarray(contract)
    return np.where(c == 0, 0, np.where((c >= 1) & (c <= 3), 1, np.where((c == 7) | (c == 9), 3, 2)))


def talon_k(contract):
    c = np.asarray(contract, np.int64)
    return np.select([np.isin(c, (1, 4)), np.isin(c, (2, 5)), np.isin(c, (3, 6))], [3, 2, 1], 0)


def bits_of(ids, valid=None):
    """OR of 1 << id over the last axis (entries where ``valid`` is False, or 0xFF, are skipped)."""
    ids = np.asarray(ids)
    ok = ids != 0xFF if valid is None else valid & (ids != 0xFF)
    b = np.where(ok, U1 << np.where(ok, ids, 0).astype(np.uint64), np.uint64(0))
    return np.bitwise_or.reduce(b, axis=-1)


def hand_dealt(perm, seat):
    """The hand of ``seat`` as dealt (Igra.razdeli: perm[12 s : 12 s + 12]) as a bitboard per game."""
    idx = 12 * np.asarray(seat, np.int64)[:, None] + np.arange(12)[None, :]
    return bits_of(np.take_along_axis(np.asarray(perm, np.int64), idx, axis=1))


def history_len(d, t):
    """n = len(zgodovina) before card play t: the plays, the ("Talon", ...) entry of an exchange and the (None, card)
    entries of Klop's revealed talon cards (Igralec.py:457 keeps them all)."""
    n = t + (np.asarray(d["group"]) != NO_PLAY).astype(np.int64)
    return n + np.where(np.asarray(d["contract"]) == 0, min(t // 4, 6), 0)


def observation(d, L, t):
    """The observation of the seat making play t, for every game (``live`` says which games have a play t).

    Returned as bitboards, from which ``dense`` builds the reference's arrays:
      opp [n,48,3]  row i, opponent o (the other three seats in seat order) -> card of that opponent's play i;
      hand [n,48]   row i of an own play -> the hand as dealt minus the own cards played before row i;
      T [n]         rows = n + (8 - n % 8);  kind [n] net type;
      talon [n,6,55] (Navadna, Solo: row j = j-th talon card, column 54 = "in the chosen group", once exchanged),
      klop_talon [n] (the talon cards revealed so far, popped from the end), king / decl [n] one-hot index (-1 none),
      discard [n] (own discards, for the declarer after an exchange), mozne [n] (the legal cards).
    """
    n = len(d["contract"])
    seat = L["seat"].astype(np.int64)
    cards = np.asarray(d["cards"], np.int64)
    contract = np.asarray(d["contract"], np.int64)
    group = np.asarray(d["group"], np.int64)
    perm = np.asarray(d["perm"], np.int64)
    live = seat[:, t] != NO_PLAY
    me = np.where(live, seat[:, t], 0)
    played = (seat != NO_PLAY) & (np.arange(48)[None, :] < t)
    bit = np.where(played, U1 << np.where(played, cards, 0).astype(np.uint64), np.uint64(0))
    own = played & (seat == me[:, None])
    opp_idx = np.where(seat < me[:, None], seat, seat - 1)
    opp = np.zeros((n, 48, 3), np.uint64)
    for o in range(3):
        opp[:, :, o] = np.where(played & ~own & (opp_idx == o), bit, 0)
    own_bits = np.where(own, bit, np.uint64(0))
    upto = np.bitwise_or.accumulate(own_bits, axis=1)
    before = upto & ~own_bits                                   # own cards are distinct
    hand = np.where(own, hand_dealt(perm, me)[:, None] & ~before, np.uint64(0))
    nh = history_len(d, t)
    kind = net_type(contract)
    k = talon_k(contract)
    talon = np.zeros((n, 6, 55), np.uint8)
    exchanged = group != NO_PLAY
    chosen = np.zeros((n, 6), bool)                            # talon card j lies in the chosen group
    for j in range(6):
        talon[exchanged, j, perm[exchanged, 48 + j]] = 1
        chosen[:, j] = exchanged & (j // np.maximum(k, 1) == group)
    talon[:, :, 54] = chosen
    shown = min(t // 4, 6)
    klop_talon = bits_of(perm[:, 54 - shown:54]) if shown else np.zeros(n, np.uint64)
    decl = np.asarray(d["declarer"], np.int64)
    king = np.asarray(d["king"], np.int64)
    mozne = bits_of(L["mozne"][:, t], np.arange(16)[None, :] < L["mozne_n"][:, t, None])
    return dict(live=live, seat=me, opp=opp, hand=hand, T=nh + (8 - nh % 8), kind=kind, talon=talon,
                klop_talon=np.where(contract == 0, klop_talon, np.uint64(0)),
                king=np.where((kind == 1) & (king < 4), king, -1),
                decl=np.where(kind == 0, -1, np.where(decl == me, 3, np.where(decl < me, decl, decl - 1))),
                discard=np.where((decl == me) & exchanged, np.asarray(d["discard_mask"], np.uint64), np.uint64(0)),
                mozne=mozne)


def unpack(b):
    """Bitboards [...] -> 0/1 uint8 [..., 54]."""
    return ((np.asarray(b, np.uint64)[..., None] >> np.arange(54, dtype=np.uint64)) & U1).astype(np.uint8)


def one_hot4(i):
    out = np.zeros(4, np.uint8)
    if i >= 0:
        out[i] = 1
    return out


def dense(o, g, with_mozne=True):
    """The reference's input list of game g (Navadna [opp, king, hand, talon, decl, discard, mozne]; Solo [opp, hand,
    talon, decl, discard, mozne]; Klop [opp, hand, talon, mozne]; Berac [opp, hand, decl, mozne]) as 0/1 uint8 arrays."""
    T, kind = int(o["T"][g]), int(o["kind"][g])
    opp = np.zeros((T, 3, 54), np.uint8)
    hand = np.zeros((T, 54), np.uint8)
    r = min(T, 48)
    opp[:r] = unpack(o["opp"][g, :r])
    hand[:r] = unpack(o["hand"][g, :r])
    talon = unpack(o["klop_talon"][g]) if kind == 0 else o["talon"][g]
    king, decl, disc = one_hot4(o["king"][g]), one_hot4(o["decl"][g]), unpack(o["discard"][g])
    out = {0: [opp, hand, talon], 1: [opp, king, hand, talon, decl, disc], 2: [opp, hand, talon, decl, disc],
           3: [opp, hand, decl]}[kind]
    return out + [unpack(o["mozne"][g])] if with_mozne else out


# ------------------------------------------------------------------ exploration (DESIGN.md section 4)
_M0, _M1, _W0, _W1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), 0x9E3779B9, 0xBB67AE85
_LO = np.uint64(0xFFFFFFFF)


def philox(seed, gid, stream, block):
    """Philox4x32-10 words [n,4] for counter (gid.lo, gid.hi, stream, block) under key = seed, vectorised over gid."""
    gid = np.asarray(gid, np.uint64)
    c0, c1 = gid & _LO, gid >> np.uint64(32)
    c2 = np.full_like(gid, np.uint64(stream))
    c3 = np.broadcast_to(np.asarray(block, np.uint64), gid.shape).copy()
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    for _ in range(10):
        p0, p1 = _M0 * c0, _M1 * c2
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ np.uint64(k0)), p1 & _LO, ((p0 >> np.uint64(32)) ^ c3 ^ np.uint64(k1)), p0 & _LO
        k0, k1 = (k0 + _W0) & 0xFFFFFFFF, (k1 + _W1) & 0xFFFFFFFF
    return np.stack([c0, c1, c2, c3], axis=-1)


def draw(word, seed, gid, idx, n):
    """Uniform in [0, n) from a Philox word: Lemire's multiply-shift, a rejected word redrawn by ``oracle.draw``."""
    word, n = np.asarray(word, np.uint64), np.asarray(n, np.uint64)
    m = word * np.maximum(n, 1)
    r = (m >> np.uint64(32)).astype(np.int64)
    reject = (m & _LO) < (np.uint64(1 << 32) % np.maximum(n, 1))
    for i in np.nonzero(reject & (n > 0))[0]:
        r[i] = O.draw(seed, int(np.ravel(gid)[i] if np.ndim(gid) else gid), ST_EXPLORE, int(np.ravel(idx)[i] if np.ndim(idx) else idx), int(n[i]))
    return r


def explores(word, random_card):
    """random.random() < random_card with random.random() = word / 2^32 for the fp32 epsilon the device receives."""
    eps = float(np.float32(random_card))
    return np.ones(np.shape(word), bool) if eps >= 1.0 else np.asarray(word, np.uint64) < np.uint64(int(eps * 2.0 ** 32))


def nth_set_bit(mask, r):
    out = np.empty(len(mask), np.int64)
    for i, (m, k) in enumerate(zip(np.asarray(mask, np.uint64).tolist(), np.asarray(r).tolist())):
        ids = [c for c in range(54) if (m >> c) & 1]
        out[i] = ids[k]
    return out


# ------------------------------------------------------------------ decisions
def first_argmax(v):
    """np.argmax along the last axis: the first NaN if there is one, else the first maximum."""
    return np.argmax(v, axis=-1)


def choose_card(q, mozne, mozne_n, t=None, seed=0, gid=None, random_card=0.0):
    """igraj_karto for one decision per row: q fp32 [n,54], mozne / mozne_n the oracle's ordered lists [n,16] / [n].
    Returns (card, qmax, explored).  next_Q_max = q[argmax card] also when the card is explored: the kernel's documented
    reading (tarok_obs.cuh), which cannot be checked against the reference here."""
    n = len(q)
    q = np.asarray(q, np.float32)
    slot = np.arange(16)[None, :] < np.asarray(mozne_n)[:, None]
    ids = np.where(slot, mozne, 0).astype(np.int64)
    vals = np.where(slot, np.take_along_axis(q, ids, axis=1).astype(np.float64), -np.inf)
    a = first_argmax(vals)
    card = np.take_along_axis(ids, a[:, None], axis=1)[:, 0]
    qmax = q[np.arange(n), card]
    explored = np.zeros(n, bool)
    if float(random_card) > 0:
        w = philox(seed, gid, ST_EXPLORE, t)
        explored = explores(w[:, 0], random_card)
        legal = bits_of(mozne, slot)
        pc = np.array([bin(int(x)).count("1") for x in legal.tolist()])
        r = draw(w[:, 1], seed, gid, 4 * t + 1, pc)
        card = np.where(explored, nth_set_bit(legal, np.where(explored, r, 0)), card)
    return card, qmax, explored


def choose_exchange(p, d, L, seed=0, gid=None, random_card=0.0, group=None):
    """menjaj_iz_talona: group = first argmax of p[54 : 54 + groups]; discards = the last k of the stable argsort of
    p[mozno_zalozit()] (NaN sorts last, so NaN cards are laid down first).  ``group`` (the one actually taken) selects
    which ``mozno_zalozit()`` list of ``L`` applies; L must come from ``oracle.lists`` run with that group.
    Returns (group, discard mask); discard 0 when fewer than k cards are discardable (Q19)."""
    n = len(p)
    p = np.asarray(p, np.float32)
    k = talon_k(d["contract"])
    groups = np.where(k > 0, 6 // np.maximum(k, 1), 0)
    gv = np.where(np.arange(6)[None, :] < groups[:, None], p[:, 54:60].astype(np.float64), -np.inf)
    want = first_argmax(gv)
    if float(random_card) > 0:
        b50 = philox(seed, gid, ST_EXPLORE, 50)
        b51 = philox(seed, gid, ST_EXPLORE, 51)
        want = np.where(explores(b50[:, 0], random_card), draw(b50[:, 1], seed, gid, 201, groups), want)
    disc = np.zeros(n, np.uint64)
    zn = L["zalozit_n"].astype(np.int64)
    for i in range(n):
        kk = int(k[i])
        if kk == 0 or zn[i] < kk:
            continue
        lst = L["zalozit"][i, :zn[i]].astype(np.int64)
        if float(random_card) > 0 and explores(b50[i, 2], random_card):
            avail = int(bits_of(lst))
            for j in range(kk):
                ids = [c for c in range(54) if (avail >> c) & 1]
                r = int(draw(b51[i:i + 1, j], seed, gid[i:i + 1], 204 + j, np.array([len(ids)]))[0])
                avail ^= 1 << ids[r]
                disc[i] |= np.uint64(1 << ids[r])
        else:
            order = np.argsort(p[i, lst].astype(np.float64), kind="stable")
            disc[i] = bits_of(lst[order[-kk:]])
    return want, disc


def targets(d, L, scores, plays, winner, qmax, factor):
    """rezultat_stiha / rezultat_igre in float64: dy [n,48,54] (NaN rows = no play), per play t of seat s in trick j:
    -70 on every card not in ``mozne``; on the played card +-vrednost_stiha(trick j) (+ if s took the trick) plus
    factor * next, next = s's next_Q_max in trick j + 1 (``qmax`` [n,48], by play) or, after s's last play, its score,
    in Berac -20 for a non-declarer when all 12 tricks were played, else +20 (Igralec.py:433-437).
    Odprti_berac is treated as Berac: the reference raises there (Q20), this follows the kernel's documented reading.
    Returns (dy, next [n,48])."""
    n = len(d["contract"])
    seat = L["seat"].astype(np.int64)
    cards = np.asarray(d["cards"], np.int64)
    contract = np.asarray(d["contract"], np.int64)
    decl = np.asarray(d["declarer"], np.int64)
    tricks = np.asarray(plays, np.int64) // 4
    dy = np.full((n, 48, 54), np.nan)
    nexts = np.zeros((n, 48))
    rows = np.arange(n)
    for t in range(48):
        j = t // 4
        on = (seat[:, t] != NO_PLAY) & (j < tricks)
        s = np.where(on, seat[:, t], 0)
        legal = unpack(bits_of(L["mozne"][:, t], np.arange(16)[None, :] < L["mozne_n"][:, t, None])).astype(bool)
        v = L["trick_value"][:, j].astype(np.float64)
        v = np.where(winner[:, j] == s, v, -v)
        nxt = np.zeros(n)
        if j + 1 < 12:
            for t2 in range(4 * (j + 1), 4 * (j + 1) + 4):
                nxt = np.where(seat[:, t2] == s, qmax[:, t2].astype(np.float64), nxt)
        final = np.asarray(scores, np.float64)[rows, s]
        berac_other = ((contract == 7) | (contract == 9)) & (s != decl)
        final = np.where(berac_other, np.where(tricks == 12, -20.0, 20.0), final)
        nxt = np.where(j + 1 < tricks, nxt, final)
        row = np.where(legal, 0.0, -70.0)
        row[rows, np.where(on, cards[:, t], 0)] = v + float(factor) * nxt
        dy[on, t] = row[on]
        nexts[:, t] = np.where(on, nxt, 0.0)
    return dy, nexts
