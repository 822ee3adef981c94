"""CPU: the C oracle (oracle/tarok_oracle.c) against vectors frozen from the REAL reference."""
import hashlib
import itertools
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN


def _replay_matches(O, g):
    r = O.replay(g["perm"], g["contract"], g["declarer"], g["king"], g["group"], g["discard_mask"], g["card"])
    assert r["err"].sum() == 0
    for k in ("seat", "mask", "winner", "scores", "plays", "hands", "piles"):
        assert (r[k] == g[k]).all(), k


def test_traces_forced(oracle, golden):
    _replay_matches(oracle, golden("traces_forced.npz"))


def test_traces_full(oracle, golden):
    _replay_matches(oracle, golden("traces_full.npz"))


def test_full_auction_dispatch(oracle, golden):
    """Igra.start: intents -> (declarer, contract, king) incl. king suit of the original intent."""
    g = golden("traces_full.npz")
    tip = np.array([-1] + [1] * 4 + [2] * 4 + [3] * 4 + [4, 5, 6, 7, 8], np.int8)
    d, c, _ = oracle.auction_fixed(tip[g["intent"]])
    assert (c == g["contract"]).all()
    assert (d[c != 0] == g["declarer"][c != 0]).all()


def test_kat_table(oracle):
    rows = json.load(open(os.path.join(GOLDEN, "kat.json")))
    assert len(rows) == 48
    n = len(rows)
    cards = np.full((n, 48), 0xFF, np.uint8)
    for i, r in enumerate(rows):
        cards[i, :len(r["cards"])] = r["cards"]
    rep = oracle.replay(
        np.array([r["perm"] for r in rows], np.uint8), [r["contract"] for r in rows],
        [r["declarer"] for r in rows], [r["king"] for r in rows], [r["group"] for r in rows],
        np.array([r["discard_mask"] for r in rows], np.uint64), cards)
    for i, r in enumerate(rows):
        assert rep["scores"][i].tolist() == r["scores"], r
        assert rep["plays"][i] == r["plays"]
    # spot values quoted in SURVEY.md A.6
    by = {(r["deal"], r["pol"], r["contract"], r["declarer"]): r for r in rows}
    assert by[("R12345", "lo", 0, 0)]["scores"] == [-17, -25, -28, 0]
    assert by[("R12345", "lo", 0, 0)]["hash"] == "493c4d1efa66fb73"
    assert by[("identity", "hi", 8, 3)]["scores"] == [0, 0, 0, 105]
    assert by[("R12345", "hi", 5, 1)]["scores"] == [0, 65, 0, 0]


def test_auction_fixed_exhaustive(oracle, golden):
    a = golden("auction_fixed.npz")
    d, c, k = oracle.auction_fixed(a["intents"])
    assert (d == a["declarer"]).all() and (c == a["contract"]).all() and (k == a["calls"]).all()
    assert a["calls"].max() <= 8
    # the hash SURVEY.md A.3 quotes for the 9 index2igra values
    lut = {tuple(int(x) for x in i): (int(dd), int(cc)) for i, dd, cc in zip(a["intents"], a["declarer"], a["contract"])}
    h = hashlib.sha256()
    for combo in itertools.product([-1, 1, 2, 3, 4, 5, 6, 7, 8], repeat=4):
        dd, cc = lut[combo]
        h.update(bytes((dd, cc * 10 + 10)))
    assert h.hexdigest()[:16] == "4c2d1393556573f9"


def test_auction_scripted_bot_model(oracle, golden):
    a = golden("auction_scripted.npz")
    d, c, k = oracle.auction_scripted(a["draws"])
    assert (d == a["declarer"]).all() and (c == a["contract"]).all() and (k == a["calls"]).all()


def test_prestej_and_cards(oracle, golden):
    u = golden("units.npz")
    v = oracle.prestej([list(r[:n]) for r, n in zip(u["pile_ids"], u["pile_len"])])
    assert (v == u["pile_val"]).all()
    full = oracle.prestej([list(range(54))])[0]
    assert full == 70
    assert (u["card_roundtrip"] == np.arange(54)).all()


def test_philox_known_answers(oracle):
    # Random123 kat_vectors for philox4x32-10
    assert oracle.philox([0, 0, 0, 0], [0, 0]) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert oracle.philox([0xffffffff] * 4, [0xffffffff] * 2) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert oracle.philox([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0]) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_synthetic_deals_are_permutations_and_uniform(oracle):
    p = oracle.deal(1234, 0, 50000)
    assert (np.sort(p, axis=1) == np.arange(54)).all()
    for s in range(4):   # hand slices ascending
        assert (np.diff(p[:, 12 * s:12 * s + 12].astype(int), axis=1) > 0).all()
    # card 0 lands in each hand with prob 12/54 and in the talon with prob 6/54
    where = np.argmax(p == 0, axis=1) // 12
    frac = np.bincount(where, minlength=5) / len(p)
    assert np.allclose(frac[:4], 12 / 54, atol=0.01) and abs(frac[4] - 6 / 54) < 0.01
    # talon order is not sorted (uniform permutation)
    asc = (np.diff(p[:, 48:].astype(int), axis=1) > 0).all(axis=1).mean()
    assert abs(asc - 1 / 720) < 0.002
    # sharding invariance: game id drives the generator
    q = oracle.deal(1234, 1000, 10)
    assert (q == p[1000:1010]).all()


def test_cpu_rollout_teacher_forced_consistency(oracle):
    """The Philox players only ever pick legal cards: replaying their trace reproduces the scores."""
    for mode in (0, 7, 16, 17, 18):
        r = oracle.rollout(99, 0, 3000, mode)
        ok = r["err"] == 0
        rep = oracle.replay(r["perm"], r["contract"], r["declarer"], r["king"], r["group"], r["discard"], r["cards"])
        assert (rep["err"][ok] == 0).all()
        assert (rep["scores"][ok] == r["scores"][ok]).all()
        assert (rep["plays"][ok] == r["plays"][ok]).all()
        assert r["stats"][8] == r["plays"].astype(np.int64).sum()



@pytest.mark.parametrize("first_gid", [2 ** 32 + 7, 1000])          # odd / even: two games share a Philox play block
@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 16])
def test_injected_rollout_reproduces_the_synthetic_one(oracle, mode, first_gid):
    """The host-buffer reference (the rows and forced contracts given, talon group 0) on what the synthetic rollout dealt
    and chose plays the same games: the two share the exchange and play-out, and differ only in where the deal and
    the contract come from."""
    n = 4000
    r = oracle.rollout(31, first_gid, n, mode)
    k = oracle.rollout_injected(31, first_gid, r["perm"], r["contract"], r["declarer"], r["king"])
    for key in ("scores", "cards", "plays", "err", "stats", "contract", "declarer", "king", "group", "discard"):
        assert (k[key] == r[key]).all(), key
    assert (k["hist"] == np.bincount(r["contract"][r["err"] == 0], minlength=10)).all()
    assert k["hist"].sum() == n - r["stats"][9]


# ---- inputs a caller can get wrong: the oracle's verdict, and the state it leaves, are defined for every byte -----------

IDENTITY = np.arange(54, dtype=np.uint8)   # seat s holds ids 12s..12s+11, the talon 48..53 in order


def _one(O, perm, contract, declarer, king=7, group=0xFF, discard=0, cards=()):
    """replay and lists of hand-built rows (one per entry of the lists)."""
    n = len(perm)
    c = np.full((n, 48), 0xFF, np.uint8)
    for i, row in enumerate(cards or [()] * n):
        c[i, :len(row)] = row
    bc = lambda x: np.broadcast_to(np.asarray(x), (n,))
    args = (np.asarray(perm, np.uint8), bc(contract).astype(np.uint8), bc(declarer).astype(np.uint8),
            bc(king).astype(np.uint8), bc(group).astype(np.uint8), bc(discard).astype(np.uint64), c)
    return O.replay(*args), O.lists(*args)


def _dealt(perm):
    hands = np.zeros(4, np.uint64)
    for s in range(4):
        for c in perm[12 * s:12 * s + 12]:
            hands[s] |= np.uint64(1 << int(c))
    talon = np.uint64(sum(1 << int(c) for c in perm[48:]))
    return hands, talon


def test_oracle_rejects_rows_that_are_not_permutations(oracle):
    """A duplicate id, an id 54..63 or an id 64..255, in a hand or in the talon, makes an error game before anything is
    dealt (k_set_deals' rule): no plays, no score, empty hands, piles and talon, empty lists -- whatever the contract."""
    rows = []
    for pos in (0, 11, 47, 48, 53):
        for bad in ("dup", 54, 63, 64, 200, 255):
            p = IDENTITY.copy()
            p[pos] = p[(pos + 1) % 54] if bad == "dup" else bad
            rows.append(p)
    n = len(rows)
    for contract, declarer, king in ((0, 0, 7), (1, 2, 1), (4, 3, 7), (7, 1, 7)):
        first = [[0] * 4] * n                                 # cards that would be legal in a valid deal
        rep, lst = _one(oracle, rows, contract, declarer, king, group=0, discard=0b111, cards=first)
        assert (rep["err"] == 1).all() and (rep["plays"] == 0).all() and (rep["scores"] == 0).all()
        assert (rep["hands"] == 0).all() and (rep["piles"] == 0).all() and (rep["talon"] == 0).all()
        assert (rep["seat"] == 0xFF).all() and (rep["mask"] == 0).all()
        assert (lst["mozne_n"] == 0).all() and (lst["zalozit_n"] == 0).all() and (lst["groups"] == 0xFF).all()
        assert (lst["seat"] == 0xFF).all()


@pytest.mark.parametrize("contract", range(10))
def test_oracle_rejects_a_declarer_above_3_for_every_contract(oracle, contract):
    """Declarer 4, 5 or 255 is an error game under every contract, Klop included (begin_contract's rule; the reference has no
    such player).  The deal stays as dealt; a valid declarer still plays."""
    dh, dt = _dealt(IDENTITY)
    rep, lst = _one(oracle, [IDENTITY] * 4, contract, [4, 5, 255, 3], king=1, group=0xFF, discard=0)
    assert rep["err"][:3].tolist() == [1, 1, 1]
    assert (rep["hands"][:3] == dh).all() and (rep["talon"][:3] == dt).all() and (rep["piles"][:3] == 0).all()
    assert (lst["mozne_n"][:3] == 0).all()
    exchange = 1 <= contract <= 6                             # declarer 3 then waits for the exchange this row does not make
    assert rep["err"][3] == (1 if exchange else 0)
    if not exchange:
        assert lst["mozne_n"][3, 0] > 0


def test_oracle_rejects_discard_bits_above_53_and_leaves_a_refused_exchange_untouched(oracle):
    """Tri (k = 3), declarer 0, talon group 0 = ids 48..50.  A discard mask with a bit in 54..63 is an invalid exchange even
    when its other bits are a valid set; so are kings, trula cards, cards of another seat or of a group not chosen, and a
    wrong count.  A refused exchange leaves hands, piles and talon as dealt; a valid one (picked-up cards included) plays."""
    dh, dt = _dealt(IDENTITY)
    b = lambda *ids: sum(1 << i for i in ids)
    cases = [
        (b(0, 1, 60), 1), (b(0, 1, 2, 54), 1), (b(0, 1, 63), 1), (b(0, 1, 2) | (1 << 63), 1),
        (b(0, 1, 7), 1),                    # the kara king
        (b(0, 1, 32), 1), (b(0, 1, 52), 1), # pagat / mond (seat 0 holds neither: also another seat's)
        (b(0, 1, 12), 1),                   # seat 1's card
        (b(0, 1, 51), 1),                   # group 1's card
        (b(0, 1), 1), (b(0, 1, 2, 3), 1), (0, 1),
        (b(0, 1, 2), 0), (b(0, 1, 48), 1),  # XVII is not discardable (Karta.vrednost 5 above VII)
        (b(5, 6, 8), 0),
    ]
    perm = [IDENTITY] * len(cases)
    rep, _ = _one(oracle, perm, 1, 0, king=1, group=0, discard=[m for m, _ in cases])
    assert rep["err"].tolist() == [e for _, e in cases]
    bad = rep["err"] == 1
    assert (rep["hands"][bad] == dh).all() and (rep["piles"][bad] == 0).all() and (rep["talon"][bad] == dt).all()
    grp0 = np.uint64(b(48, 49, 50))
    for i in np.nonzero(~bad)[0]:
        m = np.uint64(cases[i][0])
        assert rep["hands"][i, 0] == (dh[0] | grp0) & ~m and rep["piles"][i, 0] == m
        assert rep["talon"][i] == dt & ~grp0
    # groups past the last (6 / k = 2 for Tri), 7 and 255 are invalid too
    rep, _ = _one(oracle, [IDENTITY] * 3, 1, 0, king=1, group=[2, 7, 255], discard=b(0, 1, 2))
    assert (rep["err"] == 1).all() and (rep["hands"] == dh).all() and (rep["talon"] == dt).all()
