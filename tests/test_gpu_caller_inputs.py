"""GPU: the entry points of a caller that makes its own decisions -- tarok_set_deals, tarok_auction, tarok_force_contract,
tarok_exchange and tarok_step (k_step<false, POS>), the path of an external RL policy -- game by game against the C oracle
(oracle.replay / oracle.lists), with invalid inputs of every kind mixed in.

The expected values come from the oracle or from a plain numpy statement of the reference's definitions (teams from the
deal, the called king from the declarer's own intent, which card is illegal and why), never from a copy of the kernels.
A refused input leaves the game as it was, with its error bit set and stats[21] (error events) counted once; the tests
compare that state, not only the error bit.  Bar: bit-exact."""
import ctypes as C
import itertools

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SEED = 0xCA11E5
CARD_SKIP = 0xFE                              # TAROK_CARD_SKIP
ONE = np.uint64(1)
TAROKS = np.uint64(0x3FFFFF << 32)
PAGAT, MOND, SKIS = 32, 52, 53
KING_IDS = (7, 15, 23, 31)


# ---- helpers ------------------------------------------------------------------------------------------------------------

def u64(t):
    return t.detach().cpu().numpy().view(np.uint64)


def fields(env):
    import tarok_b200.env as E
    m = u64(env.meta[:env.n])
    f = lambda sh, b: ((m >> np.uint64(sh)) & np.uint64((1 << b) - 1)).astype(np.int64)
    return dict(contract=f(E.M_CONTRACT, 4), declarer=f(E.M_DECL, 2), king=f(E.M_KING, 3), team=f(E.M_TEAM, 4),
                leader=f(E.M_LEADER, 2), pos=f(E.M_POS, 2), phase=f(E.M_PHASE, 2), err=f(E.M_ERR, 1),
                plays=f(E.M_PLAYS, 6))


def same(got, want, what, rows=None):
    """Per game (first axis): got == want, on `rows` (bool mask) or all games."""
    got = np.asarray(got)
    want = np.broadcast_to(np.asarray(want), got.shape)
    bad = got != want
    if bad.ndim > 1:
        bad = bad.reshape(len(bad), -1).any(1)
    if rows is not None:
        bad &= rows
    if bad.any():
        idx = np.nonzero(bad)[0]
        raise AssertionError("%s: %d games differ, first %s (got %s, want %s)"
                             % (what, len(idx), idx[:8].tolist(), got[idx[:3]].tolist(), want[idx[:3]].tolist()))


def bits_of(ids):
    """uint64 bitboard of card ids (any shape; ids >= 54, e.g. 0xFF padding, contribute nothing) over the last axis."""
    ids = np.asarray(ids)
    v = np.where(ids < 54, np.left_shift(ONE, np.minimum(ids, 63).astype(np.uint64)), np.uint64(0))
    return np.bitwise_or.reduce(v, axis=-1)


def lowest_id(m):
    """Card id of the lowest set bit of each nonzero uint64."""
    low = m & (~m + ONE)
    return np.log2(low.astype(np.float64)).astype(np.int64)


def hands_of(perm):
    """Hands as dealt by Igra.razdeli (Igra.py:65-73), uint64 [n, 4] by seat."""
    perm = np.asarray(perm)
    return np.stack([bits_of(perm[:, 12 * s:12 * s + 12]) for s in range(4)], 1)


def device_state(env):
    n = env.n
    return dict(hands=u64(env.hands[:, :n]).T, piles=u64(env.piles[:, :n]).T, talon=u64(env.talon[:n]),
                mask=u64(env.mask[:n]), legal=u64(env.legal_mask()))


def snapshot(env):
    out = {f: getattr(env, f).clone() for f in ("meta", "hand_slots", "piles", "talon", "talon_order", "mask")}
    if env.history:
        out.update(discard=env.discard.clone(), hist=env.hist.clone())
    return out


def unchanged(before, after, what, rows=None):
    """Every field of the games in `rows` (all games, padding included, when None) is bit for bit as before."""
    for f, x in before.items():
        y = after[f]
        d = (x != y).reshape(-1, x.shape[-1]).any(0).cpu().numpy()           # per game (the last axis)
        if rows is not None:
            d = d[:len(rows)] & rows
        if d.any():
            raise AssertionError("%s: %s changed for %d games, first %s" % (what, f, d.sum(), np.nonzero(d)[0][:8].tolist()))


def intent_tables():
    """Tip code and king suit (7 = none) of every intent index tarok_auction takes: Nevronski_igralec.index2igra
    (Igralec.py:717-745) for 0..17 and the two extras of the header, 18 Odprti_berac and 19 Klop."""
    from oracle.transcript import index2igra
    tip, suit = np.empty(20, np.int8), np.full(20, 7, np.int64)
    for i in range(18):
        v, s = index2igra(i)
        tip[i] = v // 10
        if s is not None:
            suit[i] = s
    tip[18], tip[19] = 9, 0
    return tip, suit


# ---- contract start (auction / forced): oracle + the reference's definitions ----------------------------------------------

def check_contract_start(oracle, env, perm, contract, declarer, king, what):
    """The state k_begin left: against oracle.replay / oracle.lists run up to the exchange, and against the dispatch of
    Igra.start (Igra.py:38-58) and the teams of Navadna_igra.__init__ (Navadna_igra.py:20-30) stated on the deal."""
    n = env.n
    contract, declarer, king = (np.asarray(x).astype(np.int64) for x in (contract, declarer, king))
    none, zero, cards = np.full(n, 0xFF, np.uint8), np.zeros(n, np.uint64), np.full((n, 48), 0xFF, np.uint8)
    rep = oracle.replay(perm, contract, declarer, king, none, zero, cards)
    lst = oracle.lists(perm, contract, declarer, king, none, zero, cards)
    waiting = lst["groups"][:, 0, 0] != 0xFF                # the oracle split the talon: the game waits for the exchange
    err = (rep["err"] == 1) & ~waiting                      # (replay then refuses the missing exchange: not an error yet)
    m = fields(env)
    same(m["err"], err, what + ": error bits")
    same(m["phase"], 3, what + ": phase of error games", err)
    same(m["contract"], 15, what + ": contract field of error games", err)
    ok = ~err
    kg = (contract >= 1) & (contract <= 3)
    d = np.minimum(declarer, 3)
    same(m["contract"], contract, what + ": contract", ok)
    same(m["declarer"], np.where(contract == 0, 0, d), what + ": declarer", ok)
    same(m["king"], np.where(kg, king, 7), what + ": called king", ok)
    H = hands_of(perm)
    kbit = np.left_shift(ONE, (np.minimum(king, 3) * 8 + 7).astype(np.uint64))
    holders = sum(((H[:, s] & kbit) != 0).astype(np.int64) << s for s in range(4))
    solo = np.isin(contract, (4, 5, 6, 8))
    same(m["team"], np.where(kg, holders | (1 << d), np.where(solo, 1 << d, 0)), what + ": team", ok)
    same(m["leader"], np.where(np.isin(contract, (7, 9)), d, 0), what + ": leader", ok)
    same(m["phase"], np.where(waiting, 1, 2), what + ": phase", ok)
    s = device_state(env)
    want_mask = np.where(ok & ~waiting, bits_of(lst["mozne"][:, 0]), np.uint64(0))
    same(s["mask"], want_mask, what + ": mask")
    same(s["legal"], want_mask, what + ": legal_mask()")
    same(s["hands"], rep["hands"], what + ": hands")
    same(s["talon"], rep["talon"], what + ": talon")
    same(s["piles"], 0, what + ": piles")
    assert env.stats()[21] == err.sum(), what
    return err, waiting


# ---- A. deals ------------------------------------------------------------------------------------------------------------

def corrupt_row(row, kind, where, rng):
    """A row that is no permutation: a duplicate id, an id 54..63 or an id 64..255, in a hand byte or a talon byte."""
    i = int(rng.integers(0, 48)) if where == "hand" else int(rng.integers(48, 54))
    if kind == "dup":
        row[i] = row[(i + 1 + int(rng.integers(0, 53))) % 54]
    elif kind == "54-63":
        row[i] = int(rng.integers(54, 64))
    else:
        row[i] = int(rng.integers(64, 256))


@pytest.mark.parametrize("n", [1, 255, 256, 257, 511, 512, 513, 300_001])
def test_set_deals_at_every_offset_with_invalid_rows(oracle, n):
    """tarok_set_deals from byte offsets 0, 1 and 8 of a 16-byte-aligned buffer: k_set_deals stages with 16-byte loads only
    when the pointer is aligned, and n * 54 is a multiple of 16 for some of these sizes and not for others.  Invalid rows
    at the first and last row, at rows 255 / 256 (the first CTA's last row and the second's first), and (large batch) on
    1 % of the rows, of every kind, in hand and talon bytes.  Checked: error bits, stats[21], tarok_export_perm of the
    valid rows, and the valid games played to the oracle's result (forced contracts of every kind)."""
    from tarok_b200.env import TarokEnv
    rng = np.random.default_rng(n)
    perm = rng.permuted(np.tile(np.arange(54, dtype=np.uint8), (n, 1)), axis=1)
    rows = sorted({0, n - 1, 255, 256} & set(range(n)))
    if n > 1000:
        rows = sorted(set(rows) | set(rng.choice(n, n // 100, replace=False).tolist()))
    kinds = list(itertools.product(("dup", "54-63", "64-255"), ("hand", "talon")))
    for j, r in enumerate(rows):
        corrupt_row(perm[r], *kinds[j % len(kinds)], rng)
    bad = np.zeros(n, bool)
    bad[rows] = True
    contract = rng.integers(0, 10, n).astype(np.uint8)
    declarer = rng.integers(0, 4, n).astype(np.uint8)
    king = rng.integers(0, 4, n).astype(np.uint8)
    gid = 2 ** 32 + n
    env = TarokEnv(n, seed=SEED)
    buf = torch.full((n * 54 + 32,), 0xEE, dtype=torch.uint8, device="cuda")
    assert buf.data_ptr() % 16 == 0
    try:
        for off in (0, 1, 8):
            # a single-game batch: the row is invalid at offset 0 and valid at 1 and 8
            p, b = perm, bad
            if n == 1 and off:
                p, b = np.arange(54, dtype=np.uint8)[None].copy(), np.zeros(1, bool)
                rng.shuffle(p[0])
            what = "n = %d, offset %d" % (n, off)
            buf[off:off + n * 54] = torch.from_numpy(p.reshape(-1)).cuda()
            env.reset_stats()
            env._check(env._lib.tarok_set_deals(env._h, C.c_void_p(buf.data_ptr() + off), gid, env._stream()))
            m = fields(env)
            same(m["err"], b, what + ": error bits")
            same(m["phase"], np.where(b, 3, 0), what + ": phase")
            assert env.stats()[21] == b.sum(), what
            ex = env.export_perm().cpu().numpy()
            want = np.concatenate([np.sort(p[:, 12 * s:12 * s + 12], axis=1) for s in range(4)] + [p[:, 48:]], axis=1)
            same(ex, want, what + ": exported deal", ~b)
            ref = oracle.rollout_injected(SEED, gid, p, contract, declarer, king)
            env.force_contract(contract, declarer, king)
            env.exchange_synth(False)
            env.step_random(48)
            sc = env.score().cpu().numpy()
            m = fields(env)
            same(m["err"], ref["err"], what + ": error bits after play")
            same(m["plays"], ref["plays"], what + ": plays")
            same(sc, ref["scores"], what + ": scores")
            st = env.stats()
            assert (st[:21] == oracle.device_stats(ref)).all() and st[21] == ref["err"].sum(), (what, st[:22].tolist())
    finally:
        env.close()


# ---- B. auction ----------------------------------------------------------------------------------------------------------

def test_auction_every_intent_tuple_against_oracle(oracle):
    """All 20^4 = 160,000 intent tuples, one Philox deal each: contract, declarer, called king (the suit of the declarer's
    own intent for Tri/Dve/Ena, 7 otherwise), team from the deal, leader, phase, the legal mask at play 0, hands and talon
    against oracle.auction_fixed on the Tip codes and oracle.replay / oracle.lists."""
    from tarok_b200.env import TarokEnv
    tip, suit = intent_tables()
    idx = np.array(list(itertools.product(range(20), repeat=4)), np.uint8)
    n, gid = len(idx), 12345
    d, c, _ = oracle.auction_fixed(tip[idx])
    c, d = c.astype(np.int64), d.astype(np.int64)
    king = np.where((c >= 1) & (c <= 3), suit[idx[np.arange(n), d]], 7)
    env = TarokEnv(n, seed=SEED)
    try:
        env.deal(gid)
        perm = oracle.deal(SEED, gid, n)
        same(env.export_perm().cpu().numpy(), perm, "Philox deal")
        env.reset_stats()
        env.auction(idx)
        err, waiting = check_contract_start(oracle, env, perm, c, d, king, "auction")
        assert set(np.unique(c[~err]).tolist()) == set(range(10)) and waiting.sum() > 0
        # a king game whose declarer's own intent named no suit (it took another seat's level) cannot call a king
        assert err.sum() == ((king == 7) & (c >= 1) & (c <= 3)).sum()
    finally:
        env.close()


def test_auction_intents_above_19_are_error_games(oracle):
    """20,000 tuples with one to four intents in 20..255 (the rest 0..19): every game is an error game, counted once in
    stats[21], with its deal untouched and no legal card.  index2igra has no such index; before this was checked, every
    such intent was read as a Klop bid."""
    from tarok_b200.env import TarokEnv
    n, gid = 20_000, 99
    rng = np.random.default_rng(20)
    idx = rng.integers(0, 20, (n, 4))
    k = rng.integers(1, 5, n)
    for i in range(n):
        idx[i, rng.choice(4, k[i], replace=False)] = rng.integers(20, 256, k[i])
    idx[:236, 0] = np.arange(20, 256)                       # every out-of-range value at least once
    idx = idx.astype(np.uint8)
    env = TarokEnv(n, seed=SEED)
    try:
        env.deal(gid)
        perm = oracle.deal(SEED, gid, n)
        env.reset_stats()
        env.auction(idx)
        m, s = fields(env), device_state(env)
        same(m["err"], 1, "error bits")
        same(m["phase"], 3, "phase")
        same(m["contract"], 15, "contract field")
        same(s["mask"], 0, "mask")
        same(s["legal"], 0, "legal_mask()")
        same(s["hands"], hands_of(perm), "hands")
        same(s["talon"], bits_of(perm[:, 48:]), "talon")
        assert env.stats()[21] == n
    finally:
        env.close()


# ---- C. forced contracts -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("null_king", [False, True])
def test_force_contract_grid_against_oracle(oracle, null_king):
    """contract in 0..15 and 255 x declarer in 0..5 and 255 x king in 0..8 and 255 (or king_dev = NULL), six deals per
    cell: the same fields as the auction test, error games (unknown contract, declarer above 3 -- Klop included --, a
    king game without a suit) as the hardened oracle says."""
    from tarok_b200.env import TarokEnv
    kings = [None] if null_king else list(range(9)) + [255]
    cells = list(itertools.product(list(range(16)) + [255], list(range(6)) + [255], kings)) * 6
    n, gid = len(cells), 2 ** 33 + 5
    contract = np.array([x[0] for x in cells], np.uint8)
    declarer = np.array([x[1] for x in cells], np.uint8)
    king = np.array([7 if x[2] is None else x[2] for x in cells], np.uint8)
    env = TarokEnv(n, seed=SEED)
    try:
        env.deal(gid)
        perm = oracle.deal(SEED, gid, n)
        env.reset_stats()
        env.force_contract(contract, declarer, None if null_king else king)
        err, _ = check_contract_start(oracle, env, perm, contract, declarer, king, "forced, king %s" %
                                      ("NULL" if null_king else "array"))
        want = (contract > 9) | (declarer > 3) | (((contract >= 1) & (contract <= 3)) & (king > 3))
        same(err, want, "error games follow the stated rules")
    finally:
        env.close()


# ---- D. exchanges --------------------------------------------------------------------------------------------------------

EXCHANGE_CLASSES = ("valid", "count", "king", "pagat", "mond", "skis", "other seat", "other group", "bit 54-63",
                    "group 6/k", "group 7", "group 255")


def exchange_decisions(perm, contract, declarer, waiting, group0, lst, rng):
    """Per waiting game a talon group and a discard bitboard of one class of EXCHANGE_CLASSES, built from the oracle's
    mozno_zalozit() list after the pick-up of group0 and its talon groups."""
    n = len(perm)
    H = hands_of(perm)
    group, disc = group0.astype(np.uint8).copy(), np.zeros(n, np.uint64)
    cls = np.full(n, -1)
    k_of = {1: 3, 2: 2, 3: 1, 4: 3, 5: 2, 6: 1}
    for i in np.nonzero(waiting)[0]:
        k = k_of[int(contract[i])]
        z = [int(x) for x in lst["zalozit"][i, :lst["zalozit_n"][i]]]
        grp = [int(x) for x in lst["groups"][i, group0[i], :k]]
        if len(z) < k:                                      # fewer discardable cards than k: refused whatever is sent
            cls[i] = -2
            disc[i] = bits_of(np.array(z))
            continue
        c = 0 if rng.random() < 0.3 else int(rng.integers(1, len(EXCHANGE_CLASSES)))
        picked = [x for x in z if x in grp]
        first = [picked[int(rng.integers(0, len(picked)))]] if picked and rng.random() < 0.5 else []
        rest = [x for x in z if x not in first]
        base = first + [rest[j] for j in rng.permutation(len(rest))[:k - len(first)]]
        keep = base[:k - 1]
        d = int(declarer[i])
        if c == 0:
            chosen = base
        elif c == 1:
            cnt = int(rng.choice([x for x in range(5) if x != k and x <= len(z)]))
            chosen = [z[j] for j in rng.permutation(len(z))[:cnt]]
        elif c == 2:
            own = [x for x in KING_IDS if (int(H[i, d]) >> x) & 1 or x in grp]
            chosen = keep + [own[0] if own else KING_IDS[int(rng.integers(0, 4))]]
        elif c in (3, 4, 5):
            chosen = keep + [(PAGAT, MOND, SKIS)[c - 3]]
        elif c == 6:
            others = int(np.bitwise_or.reduce([H[i, s] for s in range(4) if s != d]))
            ids = [x for x in range(54) if (others >> x) & 1]
            chosen = keep + [ids[int(rng.integers(0, len(ids)))]]
        elif c == 7:
            ids = [int(x) for gg in range(6 // k) if gg != group0[i] for x in lst["groups"][i, gg, :k]]
            chosen = keep + [ids[int(rng.integers(0, len(ids)))]]
        elif c == 8:
            chosen = keep + [int(rng.integers(54, 64))]
        else:
            chosen = base
            group[i] = {9: 6 // k, 10: 7, 11: 255}[c]
        disc[i] = np.uint64(sum(1 << x for x in set(chosen)))
        cls[i] = c
    return group, disc, cls


def test_exchange_decisions_against_oracle(oracle):
    """About 100,000 games, every exchange contract (1-6), each waiting game sent one decision class: valid (from the
    oracle's mozno_zalozit list, picked-up cards included), a wrong count 0..4, a king, each trula card, a card of another
    seat, a card of a group not chosen, a bit in 54..63, or the group 6/k, 7 or 255.  The call also reaches Klop, Berac,
    Solo_brez and Odprti_berac games (some of them already playing), and error games: those come out bit for bit
    unchanged.  Every game against oracle.replay: error bit, hands by seat, piles, talon, legal mask, the discard field.
    A second call then reaches only games that are playing or erred: nothing changes at all."""
    from tarok_b200.env import TarokEnv
    n, gid = 100_003, 4242
    rng = np.random.default_rng(7)
    u = rng.random(n)
    contract = np.where(u < 0.2, rng.choice([0, 7, 8, 9], n), rng.integers(1, 7, n)).astype(np.uint8)
    declarer = np.where((u >= 0.2) & (u < 0.25), rng.integers(4, 256, n), rng.integers(0, 4, n)).astype(np.uint8)
    king = np.where((u >= 0.25) & (u < 0.27), 7, rng.integers(0, 4, n)).astype(np.uint8)
    none, zero, nocards = np.full(n, 0xFF, np.uint8), np.zeros(n, np.uint64), np.full((n, 48), 0xFF, np.uint8)
    env = TarokEnv(n, seed=SEED, history=True)
    try:
        env.deal(gid)
        perm = oracle.deal(SEED, gid, n)
        env.force_contract(contract, declarer, king)
        lst0 = oracle.lists(perm, contract, declarer, king, none, zero, nocards)
        waiting = lst0["groups"][:, 0, 0] != 0xFF
        assert set(np.unique(contract[waiting]).tolist()) == set(range(1, 7))
        # half of the games that play at once make their first card before the exchange call
        playing = lst0["mozne_n"][:, 0] > 0
        pre = playing & (rng.random(n) < 0.5)
        card0 = np.where(pre, lst0["mozne"][:, 0, 0], CARD_SKIP).astype(np.uint8)
        env.step(card0)
        env.reset_stats()
        before = snapshot(env)
        k_of = np.array([0, 3, 2, 1, 3, 2, 1, 0, 0, 0])[np.minimum(contract, 9)]
        group0 = np.where(waiting, rng.integers(0, 6, n) % np.maximum(6 // np.maximum(k_of, 1), 1), 0xFF)
        lstg = oracle.lists(perm, contract, declarer, king, group0.astype(np.uint8), zero, nocards)
        group, disc, cls = exchange_decisions(perm, contract, declarer, waiting, group0, lstg, rng)
        for c in range(len(EXCHANGE_CLASSES)):
            assert (cls == c).sum() > 1000, EXCHANGE_CLASSES[c]
        env.exchange(group, disc)
        cards = nocards.copy()
        cards[pre, 0] = card0[pre]
        rep = oracle.replay(perm, contract, declarer, king, group, disc, cards)
        lst = oracle.lists(perm, contract, declarer, king, group, disc, cards)
        same(rep["err"][cls == 0], 0, "the oracle takes every valid decision")
        same(rep["err"][cls > 0], 1, "the oracle refuses every invalid decision")
        m, s = fields(env), device_state(env)
        same(m["err"], rep["err"], "error bits")
        same(s["hands"], rep["hands"], "hands")
        same(s["piles"], rep["piles"], "piles")
        same(s["talon"], rep["talon"], "talon")
        pend = lst["mozne"][np.arange(n), rep["plays"]]
        want_mask = np.where(rep["err"] == 0, bits_of(pend), np.uint64(0))
        same(s["mask"], want_mask, "mask")
        same(s["legal"], want_mask, "legal_mask()")
        same(u64(env.discard[:n]), np.where(waiting & (rep["err"] == 0), disc, np.uint64(0)), "discard field")
        same(m["phase"], np.where(rep["err"] == 1, 3, 2), "phase", waiting)
        unchanged(before, snapshot(env), "games not waiting for an exchange", ~waiting)
        assert env.stats()[21] == (waiting & (rep["err"] == 1)).sum()
        # nobody waits any more: a second call, valid-looking or not, changes nothing
        before = snapshot(env)
        env.exchange(rng.integers(0, 256, n).astype(np.uint8), np.where(rng.random(n) < 0.5, disc, rng.integers(0, 2 ** 63, n,
                                                                                                                dtype=np.uint64)))
        unchanged(before, snapshot(env), "second exchange call")
        assert env.stats()[21] == (waiting & (rep["err"] == 1)).sum()
    finally:
        env.close()


# ---- E. cards ------------------------------------------------------------------------------------------------------------

ILLEGAL = ("follow suit", "must trump", "pagat", "other seat", "already played", "talon", "no card")
STEP_CONFIGS = [  # (name, TAROK_OPT_STEP_IMPL, lock-step, PDL)
    ("impl1", 1, True, True), ("impl1-general", 1, False, True), ("impl1-nopdl", 1, True, False),
    ("impl2", 2, True, True), ("impl3", 3, True, True), ("impl3-nopdl", 3, True, False)]
N_CARDS = 300_001


class CardRun:
    """Host-side book of one run: the oracle's games (mode, first game id), how far each game has followed the oracle's
    cards, which illegal card ended it, and the hands by seat at this point (from the oracle's post-exchange hands)."""

    def __init__(self, ref, rep0, start):
        self.ref, self.rep0 = ref, rep0
        n = len(ref["plays"])
        self.n = n
        self.rows = np.arange(n)
        self.plays = ref["plays"].astype(np.int64)
        self.ptr = np.zeros(n, np.int64)
        self.dead = np.zeros(n, bool)
        self.bad_card = np.full(n, 0xFF, np.int64)
        self.hands = start["hands"].copy()
        self.talon = start["talon"].copy()
        self.played = np.zeros(n, np.uint64)
        self.klopfam = np.isin(ref["contract"], (0, 7, 9))
        self.count = {}                                      # (what, position) -> games

    def alive(self):
        return ~self.dead & (self.ptr < self.plays)

    def advance(self, sel):
        """The games in `sel` play the oracle's next card."""
        r, t = self.rows[sel], self.ptr[sel]
        card = self.ref["cards"][r, t].astype(np.uint64)
        seat = self.rep0["seat"][r, t]
        b = np.left_shift(ONE, card)
        self.hands[r, seat] &= ~b
        self.played[r] |= b
        self.ptr[sel] += 1

    def tally(self, what, idx):
        """Count the games `idx` under `what`, by trick position."""
        c = np.bincount(self.ptr[idx] % 4, minlength=4)
        for p in range(4):
            self.count[(what, p)] = self.count.get((what, p), 0) + int(c[p])

    def illegal(self, sel, rng):
        """One illegal card for every game in `sel`, of a kind drawn per game (falling back to the next kind the game
        allows); returns (cards, kind index)."""
        r = self.rows[sel]
        t = self.ptr[r]
        pos = t % 4
        seat = self.rep0["seat"][r, t]
        hand = self.hands[r, seat]
        legal = self.rep0["mask"][r, t]
        lead = np.where(pos > 0, self.ref["cards"][r, np.maximum(t - pos, 0)], 0).astype(np.int64)
        led = np.where(lead >= 32, TAROKS, np.left_shift(np.uint64(0xFF), (lead & 24).astype(np.uint64)))
        others = np.bitwise_or.reduce(self.hands[r], axis=1) & ~hand
        cand = [
            np.where((pos > 0) & ((hand & led) != 0), hand & ~led, 0),                          # follow suit
            np.where((pos > 0) & (lead < 32) & ((hand & led) == 0) & ((hand & TAROKS) != 0),
                     hand & ~TAROKS, 0),                                                        # must trump
            np.where(self.klopfam[r] & (legal != 0) & ((legal >> np.uint64(PAGAT)) & ONE == 0),
                     hand & np.left_shift(ONE, np.uint64(PAGAT)), 0),                            # the pagat
            others,                                                                             # another seat's
            self.played[r],                                                                     # already played
            self.talon[r],                                                                      # in the talon
        ]
        cand = [c.astype(np.uint64) & ~legal for c in cand]
        kind = rng.integers(0, len(ILLEGAL), len(r))
        card = np.full(len(r), -1, np.int64)
        got = np.full(len(r), -1, np.int64)
        for step in range(len(ILLEGAL)):
            kk = (kind + step) % len(ILLEGAL)
            for j in range(len(ILLEGAL) - 1):
                s = (got < 0) & (kk == j) & (cand[j] != 0)
                if s.any():
                    m = cand[j][s]
                    m2 = m & (m - ONE)                     # the lowest or the second lowest card of the kind
                    pick = np.where((rng.random(s.sum()) < 0.5) & (m2 != 0), m2, m)
                    card[s], got[s] = lowest_id(pick), j
            s = (got < 0) & (kk == len(ILLEGAL) - 1)
            if s.any():
                x = rng.integers(54, 255, s.sum())
                card[s], got[s] = np.where(x == CARD_SKIP, 0xFF, x), len(ILLEGAL) - 1
        assert (got >= 0).all()
        return card, got


def drive_cards(env, run, rng, what):
    """The oracle's cards, corrupted per launch from the seeded schedule, with skips and random chains in between; after
    every launch the masks and the per-game plays / error bits against the book."""
    n = run.n
    pairs = np.arange(0, n - 1, 2)
    launches = 0
    while run.alive().any():
        launches += 1
        assert launches < 400, what
        alive = run.alive()
        if rng.random() < 0.15:                                            # a chain of in-kernel random steps
            c = int(rng.choice([1, 2, 3, 5]))
            env.step_random(c)
            for _ in range(c):
                run.advance(run.alive())
        else:
            skip = alive & (rng.random(n) < 0.12)
            err = alive & ~skip & (rng.random(n) < 0.006)
            u = rng.random(len(pairs))                                     # lane pairs: both, the even one, the odd one
            both, even, odd = u < 0.002, (u >= 0.002) & (u < 0.005), (u >= 0.005) & (u < 0.008)
            for sel, a, b in ((both, True, True), (even, True, False), (odd, False, True)):
                if a:
                    err[pairs[sel]] |= alive[pairs[sel]]
                if b:
                    err[pairs[sel] + 1] |= alive[pairs[sel] + 1]
            warps = np.nonzero(rng.random((n + 63) // 64) < 0.002)[0]    # whole warps (64 games of a lane block)
            for w in warps:
                err[64 * w:64 * w + 64] |= alive[64 * w:64 * w + 64]
            both_live = alive[pairs] & alive[pairs + 1]
            for a, b in ((0, 1), (1, 0)):                                  # an error next to a skip, at the trick's end
                sel = pairs[both_live & (run.ptr[pairs + a] % 4 == 3) & (rng.random(len(pairs)) < 0.003)]
                err[sel + a] = True
                err[sel + b] = False
                skip[sel + b] = True
                run.tally("error beside a skip", sel + a)
            skip &= ~err
            run.tally("whole warp", np.array([64 * w for w in warps if alive[64 * w:64 * w + 64].all()], np.int64))
            pe = err[pairs] & alive[pairs]
            po = err[pairs + 1] & alive[pairs + 1]
            run.tally("pair both", pairs[pe & po])
            run.tally("pair even alone", pairs[pe & ~po])
            run.tally("pair odd alone", pairs[~pe & po] + 1)
            card = np.full(n, 0xFF, np.int64)
            go = alive & ~skip & ~err
            card[go] = run.ref["cards"][run.rows[go], run.ptr[go]]
            card[skip] = CARD_SKIP
            bad, kind = run.illegal(err, rng)
            card[err] = bad
            for j, name in enumerate(ILLEGAL):
                run.tally(name, run.rows[err][kind == j])
            env.step(card.astype(np.uint8))
            run.dead[err] = True
            run.bad_card[err] = bad
            run.advance(go)
        m = fields(env)
        w = "%s, launch %d" % (what, launches)
        same(m["err"], run.dead | (run.ref["err"] == 1), w + ": error bits")
        same(m["plays"], run.ptr, w + ": plays")
        live = run.alive()
        want = np.where(live, run.rep0["mask"][run.rows, np.minimum(run.ptr, 47)], np.uint64(0))
        same(u64(env.mask[:n]), want, w + ": mask")
        same(u64(env.legal_mask()), want, w + ": legal_mask()")
    return launches


def check_cards_end(oracle, env, run, gid, what):
    """The oracle replays each game's card list, cut at its first illegal card; the device after score() must agree on
    every game (and the statistics over the batch)."""
    n, ref = run.n, run.ref
    cards = np.full((n, 48), 0xFF, np.uint8)
    t = np.arange(48)[None]
    cards[:] = np.where(t < run.ptr[:, None], ref["cards"], 0xFF)
    d = run.rows[run.dead]
    # 0xFF ends a card list for the oracle; for tarok_step it is an id like any other past 53
    cards[d, run.ptr[d]] = np.where(run.bad_card[d] == 0xFF, 200, run.bad_card[d])
    rep = oracle.replay(ref["perm"], ref["contract"], ref["declarer"], ref["king"], ref["group"], ref["discard"], cards)
    same(rep["err"], run.dead | (ref["err"] == 1), what + ": the oracle refuses exactly the corrupted cards")
    sc = env.score().cpu().numpy()
    m, s = fields(env), device_state(env)
    same(m["err"], rep["err"], what + ": error bits")
    same(m["plays"], rep["plays"], what + ": plays")
    hist = env.hist[:, :n].cpu().numpy().T
    played = t < rep["plays"][:, None]
    same(hist, np.where(played, (rep["seat"].astype(np.int64) << 6) | cards, 0xFF), what + ": history")
    same(s["hands"], rep["hands"], what + ": hands")
    same(s["piles"], rep["piles"], what + ": piles")
    same(s["talon"], rep["talon"], what + ": talon")
    same(sc, rep["scores"], what + ": scores")
    st = env.stats()
    ok = rep["err"] == 0
    sc64 = rep["scores"].astype(np.int64)
    player = (np.arange(4)[None] + (gid + run.rows)[:, None]) % 4
    by_player = [sc64[player == p].sum() for p in range(4)]
    want = np.concatenate([sc64.sum(0), by_player, np.bincount(ref["contract"][ok], minlength=10),
                           [ok.sum(), rep["plays"].astype(np.int64).sum(), (~ok).sum(), (~ok).sum()]])
    assert (st[:22] == want).all(), (what, st[:22].tolist(), want.tolist())


_CARD_REF = {}


def card_reference(oracle, mode, gid):
    key = (mode, gid)
    if key not in _CARD_REF:
        _CARD_REF.clear()
        ref = oracle.rollout(SEED, gid, N_CARDS, mode)
        rep0 = oracle.replay(ref["perm"], ref["contract"], ref["declarer"], ref["king"], ref["group"], ref["discard"],
                             ref["cards"])
        start = oracle.replay(ref["perm"], ref["contract"], ref["declarer"], ref["king"], ref["group"], ref["discard"],
                              np.full((N_CARDS, 48), 0xFF, np.uint8))
        assert (rep0["err"] == ref["err"]).all() and (rep0["plays"] == ref["plays"]).all()
        _CARD_REF[key] = (ref, rep0, start)
    return _CARD_REF[key]


@pytest.mark.parametrize("mode", [16, 17, 0, 7])
def test_illegal_cards_against_oracle(oracle, mode):
    """300,001 games of mode 16 / 17 / forced Klop / forced Berac at an even and an odd first game id, set up as
    oracle.rollout sets them up, driven with the oracle's cards corrupted per launch: a held card that fails to follow
    suit, a held suit card when the player must trump, the pagat in Klop/Berac while other cards are legal, another
    seat's card, a card already played, a talon card, ids 54..253 and 0xFF -- at all four trick positions, on both games
    of a lane pair and on each alone, on whole warps, next to a TAROK_CARD_SKIP at the trick-closing position, mixed with
    skips and with tarok_steps_random chains.  Every play_step configuration: impl 1 lock-step on / off, impl 2, impl 3,
    PDL on / off."""
    from tarok_b200.env import TarokEnv
    env = TarokEnv(N_CARDS, seed=SEED, history=True)
    try:
        for gid in (2 ** 33 + 2, 777):
            ref, rep0, start = card_reference(oracle, mode, gid)
            for ci, (name, impl, lock, pdl) in enumerate(STEP_CONFIGS):
                what = "mode %d gid %d %s" % (mode, gid, name)
                env.set_step_impl(impl)
                env.set_lockstep(lock)
                env.set_pdl(pdl)
                env.reset_stats()
                env.setup_synth(mode, gid)
                run = CardRun(ref, rep0, start)
                rng = np.random.default_rng([mode, gid & 1, ci])
                drive_cards(env, run, rng, what)
                check_cards_end(oracle, env, run, gid, what)
                for name_ in ILLEGAL:
                    positions = (1, 2, 3) if name_ in ("follow suit", "must trump") else (0, 1, 2, 3)
                    if name_ == "pagat" and mode not in (0, 7):
                        continue
                    for p in positions:
                        assert run.count.get((name_, p), 0) > 0, (what, name_, p)
                for name_ in ("pair both", "pair even alone", "pair odd alone", "whole warp"):
                    assert sum(run.count.get((name_, p), 0) for p in range(4)) > 0, (what, name_)
                assert run.count.get(("error beside a skip", 3), 0) > 0, what
    finally:
        env.close()
