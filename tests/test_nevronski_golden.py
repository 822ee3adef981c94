"""No GPU: the numpy restatement of the neural player (oracle/nevronski.py) reproduces what the REAL reference computed
(tests/golden/obs.npz, made by oracle/make_golden_obs.py): every observation bit, the card and next_Q_max it chose, the
exchange observation, group and discards, and the replay targets bit for bit after the cast to fp32.  This anchors the
restatement before tests/test_gpu_neural_reference.py uses it to judge the kernels."""
import numpy as np


def _games(g):
    return dict(perm=g["perm"], contract=g["contract"], declarer=g["declarer"], king=g["king"], group=g["group"],
                discard_mask=g["discard_mask"], cards=g["card"])


def test_restatement_reproduces_reference_observations_choices_and_targets(oracle, golden):
    from oracle import nevronski as N
    g = golden("obs.npz")
    d = _games(g)
    n = len(d["perm"])
    L = oracle.lists(d["perm"], d["contract"], d["declarer"], d["king"], d["group"], d["discard_mask"], d["cards"])
    idx, off, bits = g["obs_index"], g["obs_offset"], g["obs_bits"]
    row_of = {(int(r[0]), int(r[1])): k for k, r in enumerate(idx)}
    assert ((L["seat"] != 0xFF) == (g["card"] != 0xFF)).all()
    qmax = np.zeros((n, 48), np.float32)
    checked = 0
    for t in range(48):
        o = N.observation(d, L, t)
        games = np.nonzero(o["live"])[0]
        if len(games) == 0:
            continue
        ks = [row_of[(int(i), t)] for i in games]
        for i, k in zip(games, ks):
            assert (idx[k][2], idx[k][3], idx[k][4]) == (o["seat"][i], o["T"][i], o["kind"][i]), (i, t)
            flat = np.concatenate([a.reshape(-1) for a in N.dense(o, i)])
            want = np.unpackbits(bits[off[k]:off[k + 1]])[:flat.size]
            assert idx[k][5] == (flat.size + 7) // 8 and (flat == want).all(), (int(i), t)
            checked += 1
        card, qm, _ = N.choose_card(g["q"][ks], L["mozne"][games, t], L["mozne_n"][games, t])
        assert (card == g["card"][games, t]).all(), t
        assert (qm == g["qmax"][ks]).all(), t
        qmax[games, t] = qm
    assert checked == len(idx) == 2472
    # the exchange: observation (hand after the deal, talon card x group, game one-hot), group and discards
    ex = np.nonzero(g["group"] != 0xFF)[0]
    sub = {k: v[ex] for k, v in d.items()}
    Lx = {k: v[ex] for k, v in L.items()}
    grp, disc = N.choose_exchange(g["exch_p"][ex], sub, Lx)
    assert (grp == g["group"][ex]).all() and (disc == g["discard_mask"][ex]).all()
    assert (Lx["zalozit_n"] >= N.talon_k(sub["contract"])).all()
    hand = N.unpack(N.hand_dealt(sub["perm"], sub["declarer"]))
    talon = np.zeros((len(ex), 54, 6), np.uint8)
    for a in range(6):
        for j in range(3):
            c = Lx["groups"][:, a, j]
            talon[c != 0xFF, c[c != 0xFF], a] = 1
    game = np.zeros((len(ex), 15), np.uint8)
    c = sub["contract"].astype(np.int64)
    game[np.arange(len(ex)), np.where(c <= 3, (c - 1) * 4 + sub["king"], 12 + c - 4)] = 1
    flat = np.concatenate([hand, talon.reshape(len(ex), -1), game], axis=1)
    assert (flat == np.unpackbits(g["exch_obs_bits"][ex], axis=1)[:, :393]).all()
    # replay targets, factor 0.1 as in the fixture: float64 in the reference, stored as fp32
    r = oracle.replay(d["perm"], d["contract"], d["declarer"], d["king"], d["group"], d["discard_mask"], d["cards"])
    dy = N.targets(d, L, r["scores"], r["plays"], r["winner"], qmax, 0.1)[0].astype(np.float32)
    want = g["dy"]
    have = ~np.isnan(want[:, :, 0])
    assert have.sum() > 2000
    assert (dy[have].view(np.uint32) == want[have].view(np.uint32)).all()
    odprti = g["contract"] == 9                        # the reference cannot finish Odprti_berac (Q20): no golden rows
    assert (have[~odprti] == (g["card"][~odprti] != 0xFF)).all()


def test_philox_restatement_matches_the_oracle(oracle):
    from oracle import nevronski as N
    seed, gids = 0x0123456789ABCDEF, np.array([0, 1, 7, 2 ** 32 + 5, 65535], np.uint64)
    for block in (0, 13, 50, 51):
        w = N.philox(seed, gids, 8, block)
        for i, gid in enumerate(gids.tolist()):
            want = oracle.philox([gid & 0xFFFFFFFF, gid >> 32, 8, block], [seed & 0xFFFFFFFF, seed >> 32])
            assert w[i].tolist() == want
    for n_ in (1, 3, 11, 12, 53):
        for idx in (1, 9, 201, 204):
            w = N.philox(seed, gids, 8, idx >> 2)[:, idx & 3]
            got = N.draw(w, seed, gids, idx, np.full(len(gids), n_))
            assert got.tolist() == [oracle.draw(seed, int(x), 8, idx, n_) for x in gids.tolist()]
