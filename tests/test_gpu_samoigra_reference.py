"""GPU: whole ``Samoigra`` rollouts (tarok_b200/samoigra.py) judged decision by decision against the float64 host
restatement of the reference's neural player (oracle/nevronski.py) and the mixed-table oracle (oracle/mixed.c).

The players' networks are the parameter-free stand-ins of oracle/stub_nets.py: their outputs are small integers, exact in
fp32, bf16 and fp16, that depend on every input tensor, on the row order counted from the end, on the player and (through a
final ``mod m``) tie often.  So every decision has one right answer, with no tolerance:

  * deal: ``hands0`` / ``talon_order`` against ``oracle.deal``;
  * bids: each player's ``Vrednotenje_roke`` in float64 on the dealt hand of that player's seat, argmax, and the exploration
    of ``odigraj`` reproduced with a generator of the test's own (same device, seed and calls, continued across rollouts);
    the intents handed to ``env.auction`` must be these;
  * auction, king, the bots' exchanges and cards, scores: ``mixed.replay_bots`` on the device's cards;
  * exchanges of neural declarers: the exchange observation built from the deal, the declarer's player's ``Zalaganje`` in
    float64, ``choose_exchange`` at that player's epsilon -- group and discards exact, Q19 hands error games on both sides;
  * cards: teacher-forced on the device's history, the observation of every play, the mover's player's net for the game's
    type in float64, ``choose_card`` at that player's epsilon -- card and qmax exact;
  * statistics: the per-player sums, finished / error games and plays;
  * ``vzorci``: keys, order, observations and replay targets of every neural play, and none of a bot.

Configurations: four distinct players at eps [0, 0.05, 0.3, 1] in fp32 / bf16 / fp16 with a second ``odigraj`` on the same
object at a game id above 2^32; two bots beside two neural players (a ragged batch in bf16); one bot; one shared player."""
import time

import numpy as np
import pytest
import torch

import tarok_b200.env as E
from oracle import mixed
from oracle import nevronski as N
from oracle import oracle as O
from oracle import stub_nets as S

pytestmark = pytest.mark.gpu

SEED = 0x5A3016A7E5
FACTOR = 0.3
NET = {0: "Klop", 1: "Navadna_igra", 2: "Solo", 3: "Berac"}
CHUNK = 1024                                             # games per float64 forward on the host


def u64(t):
    return t.detach().cpu().numpy().view(np.uint64)


def _u32(x):
    return np.ascontiguousarray(x, np.float32).view(np.uint32)


class _Judge:
    """A Samoigra with its calls to ``env.auction`` / ``env.exchange`` recorded, and the host's copy of its bid-exploration
    generator."""

    def __init__(self, n, mreze, random_card, dtype, boti=()):
        from tarok_b200.samoigra import Samoigra
        self.s = Samoigra(n, mreze=mreze, seed=SEED, random_card=random_card, dtype=dtype, boti=boti)
        self.host_nets = mreze if isinstance(mreze, list) else [mreze]          # the same modules, run on CPU in float64
        self.gen = torch.Generator(device=self.s.dev)
        self.gen.manual_seed(SEED & 0x7FFFFFFFFFFFFFFF)
        self.calls = {}
        env = self.s.env
        auction, exchange = env.auction, env.exchange

        def rec_auction(intents, bots=None):
            self.calls["intents"] = intents.cpu().numpy().copy()
            self.calls["bots"] = None if bots is None else bots.cpu().numpy().copy()
            return auction(intents, bots=bots)

        def rec_exchange(group, discard, bots=None):
            self.calls["group"] = group.cpu().numpy().copy()
            self.calls["discard"] = u64(discard).copy()
            return exchange(group, discard, bots=bots)

        env.auction, env.exchange = rec_auction, rec_exchange

    def close(self):
        self.s.zapri()


def _explore_check(explored, eps, what):
    m = explored.size
    if eps == 0.0 or eps == 1.0:
        assert explored.all() if eps == 1.0 else not explored.any(), what
    else:
        assert abs(explored.mean() - eps) <= 5 * np.sqrt(eps * (1 - eps) / m) + 1e-9, (what, explored.mean(), eps)


def _pack(x):
    """Device 0/1 fp32 [..., 54] -> bitboards on the host; asserts every entry is 0 or 1."""
    assert bool(((x == 0) | (x == 1)).all())
    w = torch.ones(1, dtype=torch.int64, device=x.device) << torch.arange(54, device=x.device)
    return (x.to(torch.int64) * w).sum(-1).cpu().numpy().view(np.uint64)


def _check_sample(o, games, kind, T, stanje):
    """The replay sample's input list (no legal-mask vector) == the observation of its play, element for element."""
    names = {0: ["opp", "hand", "talon"], 1: ["opp", "king", "hand", "talon", "decl", "disc"],
             2: ["opp", "hand", "talon", "decl", "disc"], 3: ["opp", "hand", "decl"]}[kind]
    assert len(stanje) == len(names)
    B, r = len(games), min(T, 48)
    for name, a in zip(names, stanje):
        if name in ("opp", "hand"):
            m = _pack(a).reshape((B, T, 3) if name == "opp" else (B, T))
            assert (m[:, :r] == o[name][games, :r]).all() and (m[:, r:] == 0).all(), name
        elif name == "talon" and kind == 0:
            assert (_pack(a) == o["klop_talon"][games]).all(), name
        elif name == "talon":
            assert (a.cpu().numpy() == o["talon"][games]).all(), name
        elif name in ("king", "decl"):
            idx = o[name][games]
            want = ((idx[:, None] == np.arange(4)[None, :]) & (idx[:, None] >= 0)).astype(np.float32)
            assert (a.cpu().numpy() == want).all(), name
        else:
            assert (_pack(a) == o["discard"][games]).all(), name


def _rollout(j, first_gid):
    """One ``odigraj`` at ``first_gid``, every decision judged.  Returns counts for the report."""
    s, n, seed = j.s, j.s.n, j.s.env.seed
    env = s.env
    P, boti = s.igralci, s.boti
    eps = [float(x) for x in s.random_card]
    t0 = time.perf_counter()
    st, _ = s.odigraj(first_game_id=first_gid)
    torch.cuda.synchronize()
    t_dev = time.perf_counter() - t0
    rep = dict(bids=0, bids_explored=0, exchanges=0, exchanges_explored=0, cards=0, cards_tied=0, cards_explored=0)
    gid = np.arange(n, dtype=np.uint64) + np.uint64(first_gid)
    rot = ((np.arange(4)[None, :] + (gid % np.uint64(4)).astype(np.int64)[:, None]) & 3)     # player of seat s, (s + gid) % 4
    player = rot if P == 4 else np.zeros_like(rot)
    bot_seat = np.isin(player, sorted(boti))
    botmask = (bot_seat * (1 << np.arange(4))).sum(1).astype(np.uint8)
    rows = np.arange(n)

    # ---- deal
    perm = O.deal(seed, first_gid, n)
    h0 = u64(env.hands0[:, :n])
    for seat in range(4):
        assert (h0[seat] == N.hand_dealt(perm, np.full(n, seat))).all(), seat
    order = u64(env.talon_order[:n])
    for k in range(6):
        assert ((order >> np.uint64(6 * k)) & np.uint64(63) == perm[:, 48 + k]).all(), k

    # ---- bids: Vrednotenje_roke of the seat's player on the dealt hand, argmax; exploration from the host generator
    want = np.zeros((n, 4), np.int64)
    for seat in range(4):
        hand = N.unpack(N.hand_dealt(perm, np.full(n, seat)))
        for p in range(P):
            g = np.nonzero((player[:, seat] == p) & ~bot_seat[:, seat])[0]
            if len(g):
                want[g, seat] = np.argmax(S.host(j.host_nets[p]["Vrednotenje_roke"], hand[g]), axis=1)
    explored = np.zeros((n, 4), bool)
    if max(eps) > 0:
        r = torch.rand((n, 4), device=s.dev, generator=j.gen).cpu().numpy()
        drawn = torch.randint(0, 18, (n, 4), device=s.dev, generator=j.gen).cpu().numpy()
        explored = r < np.asarray(eps, np.float32)[player]
        want = np.where(explored, drawn, want)
    assert np.array_equal(j.calls["intents"], want), "bid intents"
    assert (j.calls["bots"] is None) == (not boti)
    if boti:
        assert np.array_equal(j.calls["bots"], botmask), "bot seat masks"
    for p in set(range(P)) - set(boti):
        mine = (player == p) & ~bot_seat
        _explore_check(explored[mine], np.float32(eps[p]), ("bids", p))
        rep["bids"] += int(mine.sum())
        rep["bids_explored"] += int(explored[mine].sum())

    # ---- the whole game through the mixed-table oracle, on the device's exchanges and cards
    meta = u64(env.meta[:n])
    field = lambda sh, b: ((meta >> np.uint64(sh)) & np.uint64((1 << b) - 1)).astype(np.int64)
    hist = env.hist[:, :n].cpu().numpy().T
    cards = np.where(hist == 0xFF, 0xFF, hist & 63).astype(np.uint8)
    grp, disc = j.calls["group"], j.calls["discard"]
    ref = mixed.replay_bots(seed, first_gid, perm, want, botmask, grp, disc, cards)
    err = field(E.M_ERR, 1)
    assert (ref["mismatch"] == -1).all(), "bot cards"
    assert np.array_equal(ref["err"], err), "error games"
    contract, decl, king = (ref[k].astype(np.int64) for k in ("contract", "declarer", "king"))
    assert np.array_equal(contract, field(E.M_CONTRACT, 4)), "contract"
    assert np.array_equal(decl, field(E.M_DECL, 2)), "declarer"
    assert np.array_equal(king, field(E.M_KING, 3)), "king"
    ok = err == 0
    assert np.array_equal(ref["plays"][ok], cards[ok]), "plays"
    assert (cards[~ok] == 0xFF).all()
    assert np.array_equal(ref["scores"], env.scores[:n].cpu().numpy()), "scores"
    dev_group = field(E.M_GROUP, 3)
    done = ok & (ref["group"] != 0xFF)
    assert np.array_equal(ref["group"][done], dev_group[done]) and np.array_equal(ref["discard"][done], u64(env.discard[:n])[done])

    # ---- exchanges of the neural declarers
    k = N.talon_k(contract)
    owner = player[rows, decl]
    neural_ex = (k > 0) & ~bot_seat[rows, decl]
    assert (grp[~neural_ex] == 0xFF).all() and (disc[~neural_ex] == 0).all()
    for p in set(range(P)) - set(boti):
        g = np.nonzero(neural_ex & (owner == p))[0]
        if not len(g):
            continue
        x = N.exchange_observation(perm[g], contract[g], decl[g], king[g])
        q = S.host(j.host_nets[p]["Zalaganje"], x).astype(np.float32)
        sub = dict(perm=perm[g], contract=contract[g], declarer=decl[g], king=king[g], group=grp[g], discard_mask=disc[g],
                   cards=np.full((len(g), 48), 0xFF, np.uint8))
        Lx = O.lists(*[sub[f] for f in ("perm", "contract", "declarer", "king", "group", "discard_mask", "cards")])
        want_g, want_d = N.choose_exchange(q, sub, Lx, seed, gid[g], eps[p])
        assert np.array_equal(want_g, grp[g]), ("exchange group", p)
        assert np.array_equal(want_d, disc[g]), ("exchange discards", p)
        q19 = Lx["zalozit_n"] < k[g]
        assert np.array_equal(err[g].astype(bool), q19), ("Q19", p)
        rep["exchanges"] += len(g)
        if 0 < eps[p]:
            rep["exchanges_explored"] += int(N.explores(N.philox(seed, gid[g], N.ST_EXPLORE, 50)[:, 0], eps[p]).sum())

    # ---- statistics
    fin = ref["err"] == 0
    sc = ref["scores"].astype(np.int64)
    for p in range(4):
        assert st[E.S_PLAYER + p] == (sc * (rot == p))[fin].sum(), ("stats player", p)
    assert st[E.S_FINISHED] == fin.sum() and st[E.S_ERRORS] == (~fin).sum()
    assert st[E.S_STEPS] == (ref["plays"] != 0xFF).sum()

    # ---- cards (teacher-forced on the device history) and the replay samples, play by play
    d = dict(perm=perm, contract=contract, declarer=decl, king=king, group=ref["group"], discard_mask=ref["discard"],
             cards=cards)
    L = O.lists(perm, contract, decl, king, ref["group"], ref["discard"], cards)
    played = cards != 0xFF
    assert (hist[played] >> 6 == L["seat"][played]).all()
    qmax = env.qmax_hist[:, :n].cpu().numpy().T.copy()
    seat_all = np.where(played, L["seat"], 0).astype(np.int64)
    neural_play = played & ~np.take_along_axis(bot_seat, seat_all, axis=1)
    qmax[~neural_play] = 0                       # a bot's play records nothing a neural target may read
    R = O.replay(perm, contract, decl, king, ref["group"], ref["discard"], cards, want_state=False)
    dy_ref, nxt = N.targets(d, L, R["scores"], R["plays"], R["winner"], qmax, FACTOR)
    samples = s.vzorci(FACTOR, first_gid)
    n_samples = 0
    for t in range(48):
        if not played[:, t].any():
            break
        o = N.observation(d, L, t)
        assert np.array_equal(o["live"] & ok, played[:, t]), t
        pl = player[rows, o["seat"]]
        key = np.where(neural_play[:, t], pl * 256 + o["kind"] * 64 + o["T"], -1)
        for kk in np.unique(key[key >= 0]):
            games = np.nonzero(key == kk)[0]
            p, kind, T = int(kk) // 256, (int(kk) % 256) // 64, int(kk) % 64
            for a in range(0, len(games), CHUNK):
                g = games[a:a + CHUNK]
                q = S.host(j.host_nets[p][NET[kind]], N.dense_batch(o, g, with_mozne=False)).astype(np.float32)
                mz, mzn = L["mozne"][g, t], L["mozne_n"][g, t]
                card, qm, ex = N.choose_card(q, mz, mzn, t, seed, gid[g], eps[p])
                bad = np.nonzero(card != cards[g, t])[0]
                assert len(bad) == 0, ("card", t, p, NET[kind], T, g[bad[:5]].tolist(), card[bad[:5]].tolist(),
                                       cards[g[bad[:5]], t].tolist())
                assert (_u32(qm) == _u32(qmax[g, t])).all(), ("qmax", t, p)
                slot = np.arange(16)[None, :] < mzn[:, None]
                v = np.where(slot, np.take_along_axis(q, np.where(slot, mz, 0).astype(np.int64), axis=1), -np.inf)
                rep["cards_tied"] += int(((v == v.max(1, keepdims=True)).sum(1) > 1).sum())
                rep["cards_explored"] += int(ex.sum())
                rep["cards"] += len(g)
            # the replay sample of this (player, net, T) at play t
            sp, ime, sT, stanje, dy = next(samples)
            assert (sp, ime, sT) == (p, NET[kind], T), (t, (sp, ime, sT), (p, NET[kind], T))
            assert dy.shape == (len(games), 54)
            _check_sample(o, games, kind, T, stanje)
            dy = dy.cpu().numpy().astype(np.float64)
            want_dy = dy_ref[games, t]
            c = cards[games, t].astype(np.int64)
            other = np.ones_like(dy, bool)
            other[np.arange(len(games)), c] = False
            assert np.array_equal(dy[other], want_dy[other]), ("targets -70 / 0", t)
            have, want_c = dy[np.arange(len(games)), c], want_dy[np.arange(len(games)), c]
            v, nx = np.abs(L["trick_value"][games, t // 4].astype(np.float64)), nxt[games, t]
            tol = 2.0 ** -23 * (v + np.abs(FACTOR * nx)) + np.abs(nx) * abs(float(np.float32(FACTOR)) - FACTOR)
            assert (np.abs(have - want_c) <= tol).all(), ("target of the played card", t)
            n_samples += len(games)
    assert next(samples, None) is None, "vzorci yields more than the neural plays"
    assert n_samples == neural_play.sum() == rep["cards"]
    if P == 4 and not boti:
        assert n_samples == st[E.S_STEPS]
    rep.update(rollout_ms=round(1e3 * t_dev, 1), judge_s=round(time.perf_counter() - t0 - t_dev, 1),
               errors=int((~fin).sum()), bots=sorted(boti))
    return rep


def _report(name, rep):
    c = max(rep["cards"], 1)
    print("%s: %d bids (%.3f explored), %d exchanges (%.3f explored), %d cards (%.3f tied at the top, %.3f explored), "
          "%d error games; odigraj %.1f ms, judged in %.1f s" % (
              name, rep["bids"], rep["bids_explored"] / max(rep["bids"], 1), rep["exchanges"],
              rep["exchanges_explored"] / max(rep["exchanges"], 1), rep["cards"], rep["cards_tied"] / c,
              rep["cards_explored"] / c, rep["errors"], rep["rollout_ms"], rep["judge_s"]))


@pytest.mark.parametrize("dtype", ["float32", "bfloat16", "float16"])
def test_four_distinct_players(dtype):
    """Config A: four distinct stub players at eps 0 / 0.05 / 0.3 / 1; a second odigraj on the same object (arenas,
    qmax_hist and the bid generator carried over) at a first game id above 2^32."""
    j = _Judge(8192, [S.nets(p) for p in range(4)], [0.0, 0.05, 0.3, 1.0], getattr(torch, dtype))
    for first_gid in (0, 2 ** 32 + 3):
        rep = _rollout(j, first_gid)
        assert rep["cards"] > 20 * 8192 and rep["cards_tied"] > 0.05 * rep["cards"]
        _report("A %s gid %d" % (dtype, first_gid), rep)
    j.close()


@pytest.mark.parametrize("dtype,n", [("float32", 8192), ("bfloat16", 8191)])
def test_two_bots_beside_two_players(dtype, n):
    """Config B: bots are players 1 and 3 (their epsilons are set and must be ignored), stub players 0 and 2 at eps 0.1
    and 0.2; game ids 1 then 2 on the same object; the bf16 batch is ragged."""
    j = _Judge(n, [S.nets(0), None, S.nets(2), None], [0.1, 0.6, 0.2, 0.9], getattr(torch, dtype), boti=(1, 3))
    for first_gid in (1, 2):
        rep = _rollout(j, first_gid)
        assert rep["cards"] > 10 * n
        _report("B %s n %d gid %d" % (dtype, n, first_gid), rep)
    j.close()


def test_one_bot():
    """Config C: player 0 is a bot, three stub players; an odd first game id."""
    j = _Judge(8192, [None, S.nets(1), S.nets(2), S.nets(3)], [0.5, 0.05, 0.1, 0.3], torch.float32, boti=(0,))
    rep = _rollout(j, 1001)
    _report("C float32 gid 1001", rep)
    j.close()


def test_one_shared_player():
    """Config D: igralci = 1, one stub set plays every seat at eps 0.15."""
    j = _Judge(8192, S.nets(2), 0.15, torch.float32)
    assert j.s.igralci == 1
    rep = _rollout(j, 6)
    _report("D float32 gid 6", rep)
    j.close()
