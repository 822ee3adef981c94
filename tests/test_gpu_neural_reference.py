"""GPU: the neural self-play kernels (tarok_b200/csrc/tarok_obs.cuh) against the float64 host restatement of the
reference's neural player (oracle/nevronski.py, itself pinned to the real reference by tests/test_nevronski_golden.py).

Games are set up from the C oracle's deal, contract and exchange for a mode and seed, then driven by the DEVICE's own
choices from seeded network outputs q.  After each game (or each step) the device history is replayed through the
oracle with teacher forcing, and every decision -- observation, card, next_Q_max, exploration, exchange, replay
target -- is judged against the restatement.  Both game-id parities are used (the player of seat s is (s + gid) % 4)."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SEED = 0x5EED0042AB
FLT_MAX = np.finfo(np.float32).max
REGIMES = ("ties", "zeros", "wide", "neg_inf", "nan_one", "all_nan")


def _q(rng, regime, n, legal):
    """fp32 [n,54] network outputs of one regime; `legal` (uint64 [n]) places the NaN of "nan_one" on a legal card."""
    if regime == "ties":
        return rng.integers(0, 3, (n, 54)).astype(np.float32)
    if regime == "zeros":
        return np.where(rng.random((n, 54)) < 0.5, np.float32(0.0), np.float32(-0.0)).astype(np.float32)
    if regime in ("wide", "nan_one"):
        e = rng.integers(-149, 128, (n, 54)).astype(np.float64)            # subnormals up to 2^127
        q = (np.ldexp(rng.random((n, 54)) + 0.5, e.astype(np.int32)) * rng.choice([-1.0, 1.0], (n, 54)))
        q = np.clip(q, -FLT_MAX, FLT_MAX).astype(np.float32)
        pick = rng.random((n, 54))
        q[pick < 0.05] = FLT_MAX
        q[pick > 0.95] = -FLT_MAX
        q[(pick > 0.4) & (pick < 0.45)] = rng.integers(-3, 3, int(((pick > 0.4) & (pick < 0.45)).sum()))  # ties among ordinary values
        if regime == "nan_one":                                               # one NaN on a random legal card
            bits = ((np.asarray(legal, np.uint64)[:, None] >> np.arange(54, dtype=np.uint64)) & np.uint64(1)).astype(bool)
            cnt = bits.sum(1)
            r = (rng.random(n) * np.maximum(cnt, 1)).astype(np.int64)
            pick = np.argmax(bits & (np.cumsum(bits, 1) == r[:, None] + 1), axis=1)
            q[np.nonzero(cnt)[0], pick[cnt > 0]] = np.nan
        return q
    if regime == "neg_inf":
        q = np.full((n, 54), -np.inf, np.float32)
        q[rng.random(n) < 0.3] = -FLT_MAX                                     # below the kernels' old start value too
        return q
    if regime == "all_nan":
        return np.full((n, 54), np.nan, np.float32)
    raise ValueError(regime)


def _setup(n, mode, first_gid, history=True, exchange=True):
    import torch  # noqa: F401
    from oracle import oracle as O
    from tarok_b200.env import TarokEnv
    r = O.rollout(SEED, first_gid, n, mode)
    env = TarokEnv(n, seed=SEED, history=history)
    env.set_deals(r["perm"], first_gid)
    env.force_contract(r["contract"], r["declarer"], r["king"])
    if exchange:
        env.exchange(r["group"], r["discard"])
    d = dict(perm=r["perm"], contract=r["contract"], declarer=r["declarer"], king=r["king"], group=r["group"],
             discard_mask=r["discard"], cards=np.full((n, 48), 0xFF, np.uint8))
    return env, d


def _lists(d):
    from oracle import oracle as O
    return O.lists(d["perm"], d["contract"], d["declarer"], d["king"], d["group"], d["discard_mask"], d["cards"])


def _u32(x):
    return np.ascontiguousarray(x, np.float32).view(np.uint32)


def _select_ptr_table(env, n_total, q_by_key, eps4, cards, qmax):
    """tarok_select_action_buckets: the table of bucket outputs as 128 DEVICE pointers."""
    import torch
    sel, cnt, _, selkey = env._bk[:4]
    tab = torch.zeros(128, dtype=torch.int64)
    for k, q in q_by_key.items():
        tab[k] = q.data_ptr()
    tab = tab.to(env.torch_device)
    eps = (C.c_float * 4)(*[float(x) for x in eps4])
    p = lambda t: C.c_void_p(t.data_ptr())
    env._check(env._lib.tarok_select_action_buckets(env._h, p(tab), p(sel), p(selkey), p(cnt), int(n_total), eps, p(cards),
                                                    p(qmax), env._stream()))


def _play(env, d, regime, eps, variant, rng):
    """Drives every game to its end with the device's choices; returns per play the q rows, device cards / qmax and
    legal masks."""
    import torch
    n = env.n
    dev = env.torch_device
    qs = np.zeros((n, 48, 54), np.float32)
    card = np.full((n, 48), 0xFF, np.uint8)
    qmax = np.zeros((n, 48), np.float32)
    mask = np.zeros((n, 48), np.uint64)
    eps4 = [eps] * 4
    for t in range(48):
        live = env.live().cpu().numpy()
        if not live.any():
            break
        legal = env.mask[:n].cpu().numpy().view(np.uint64)
        q = _q(rng, regime, n, legal)
        cards = torch.full((env.n_alloc,), 0xFF, dtype=torch.uint8, device=dev)
        qm = torch.zeros(n, dtype=torch.float32, device=dev)
        if variant == "plain":
            sel = np.nonzero(live)[0].astype(np.int32)
            env.select_action(torch.from_numpy(q[sel]), sel, eps, cards, qm)
        else:
            sel_dev, cnt = env.obs_buckets(4)
            total = int(cnt[255])
            order = sel_dev[:total].long().cpu().numpy()
            qd = torch.from_numpy(q).to(dev)
            q_by_key = {k: qd[torch.from_numpy(order[cnt[128 + k]:cnt[128 + k] + cnt[k]]).to(dev)].contiguous()
                        for k in range(127) if cnt[k]}
            if variant == "tab":
                env.select_action_buckets(total, q_by_key, eps4, cards, qm)
            else:
                _select_ptr_table(env, total, q_by_key, eps4, cards, qm)
        c = cards[:n].cpu().numpy()
        qs[:, t] = q
        card[live, t] = c[live]
        qmax[live, t] = qm.cpu().numpy()[live]
        mask[live, t] = legal[live]
        env.step(cards)
    torch.cuda.synchronize()
    return qs, card, qmax, mask


def _judge_cards(env, d, L, qs, card, qmax, mask, eps, first_gid):
    """Every decision of every game against the restatement: card exactly (argmax or explored), qmax bit for bit
    (NaN as NaN), the device legal mask against the oracle's ``mozne``."""
    from oracle import nevronski as N
    n = env.n
    gid = np.arange(n, dtype=np.uint64) + np.uint64(first_gid)
    decided, explored = 0, 0
    qmax_ref = np.zeros((n, 48), np.float32)
    for t in range(48):
        on = card[:, t] != 0xFF
        assert (on == (L["seat"][:, t] != 0xFF)).all(), t
        if not on.any():
            continue
        g = np.nonzero(on)[0]
        legal = N.bits_of(L["mozne"][g, t], np.arange(16)[None, :] < L["mozne_n"][g, t, None])
        assert (legal == mask[g, t]).all(), t
        c, qm, ex = N.choose_card(qs[g, t], L["mozne"][g, t], L["mozne_n"][g, t], t, env.seed, gid[g], eps)
        bad = np.nonzero(c != card[g, t])[0]
        assert len(bad) == 0, ("card", t, g[bad[:5]].tolist(), c[bad[:5]].tolist(), card[g[bad[:5]], t].tolist())
        assert (_u32(qm) == _u32(qmax[g, t])).all(), ("qmax", t)
        qmax_ref[g, t] = qm
        decided += len(g)
        explored += int(ex.sum())
    return decided, explored, qmax_ref


@pytest.mark.parametrize("variant", ["plain", "tab", "ptr"])
@pytest.mark.parametrize("regime", REGIMES)
def test_card_choice_matches_restatement(regime, variant):
    """igraj_karto through tarok_select_action, the by-value bucket table and the device pointer table, for every
    q regime, at eps 0 / 0.3 / 1.0: no game may turn into an error game, and every card and qmax is the restatement's."""
    n, mode = 4096, 17
    rng = np.random.default_rng(REGIMES.index(regime) * 3 + ["plain", "tab", "ptr"].index(variant))
    for eps, first_gid in ((0.0, 0), (0.3, 1), (1.0, 2)):
        env, d = _setup(n, mode, first_gid)
        errors0 = env.errors()
        qs, card, qmax, mask = _play(env, d, regime, eps, variant, rng)
        assert env.errors() == errors0, "a legal decision turned a game into an error game"
        d["cards"] = card
        hist = env.hist[:, :n].cpu().numpy().T
        assert ((hist & 63) == card)[card != 0xFF].all()
        L = _lists(d)
        decided, explored, _ = _judge_cards(env, d, L, qs, card, qmax, mask, eps, first_gid)
        assert decided > 20 * (n - errors0)
        if eps == 1.0:
            assert explored == decided
        elif eps == 0.3:
            assert 0.27 < explored / decided < 0.33
        env.close()


def test_no_history_env_breaks_pickup_ties_like_the_reference():
    """Without history (no hands as dealt on the device) a declarer following suit with a dealt card and a card picked up
    from the talon of equal q must still take the dealt one first (list order), exactly as with history."""
    import torch
    from oracle import nevronski as N
    n = 65536
    res = []
    for history in (True, False):
        env, d = _setup(n, 16, 1, history=history)
        card = np.full((n, 48), 0xFF, np.uint8)
        qs = np.zeros((n, 48, 54), np.float32)
        for t in range(48):
            live = env.live().cpu().numpy()
            if not live.any():
                break
            q = np.zeros((n, 54), np.float32)                                # every legal card ties
            cards, _ = env.select_action(torch.from_numpy(q))
            card[live, t] = cards[:n].cpu().numpy()[live]
            env.step(cards)
        d["cards"] = card
        L = _lists(d)
        for t in range(48):
            g = np.nonzero(card[:, t] != 0xFF)[0]
            c, _, _ = N.choose_card(qs[g, t], L["mozne"][g, t], L["mozne_n"][g, t])
            assert (c == card[g, t]).all(), (history, t)
        res.append(card)
        env.close()
    assert (res[0] == res[1]).all()
    # the ties that matter were met: a declarer's list in which a picked-up card follows a dealt one of the same suit
    assert (L["mozne"][:, :, 1:] < L["mozne"][:, :, :-1]).any()


def _targets_check(env, d, L, qmax_ref, factor):
    from oracle import nevronski as N
    from oracle import oracle as O
    n = env.n
    r = O.replay(d["perm"], d["contract"], d["declarer"], d["king"], d["group"], d["discard_mask"], d["cards"])
    dy, seat, _ = env.targets(final_reword_factor=factor)
    dy, seat = dy.cpu().numpy(), seat.cpu().numpy()
    ref, nxt_all = N.targets(d, L, r["scores"], r["plays"], r["winner"], qmax_ref, factor)
    played = ~np.isnan(ref[:, :, 0])
    assert (seat[played] == L["seat"][played]).all() and (seat[~played] == 0xFF).all()
    assert (dy[~played] == 0).all()
    assert np.array_equal(dy[played] == -70.0, ref[played] == -70.0)
    # on the played card: value + factor * next, fp32 on the device, float64 here
    g, t = np.nonzero(played)
    c = d["cards"][g, t].astype(np.int64)
    have, want = dy[g, t, c].astype(np.float64), ref[g, t, c]
    v, nxt = np.abs(L["trick_value"][g, t // 4].astype(np.float64)), nxt_all[g, t]
    tol = 2.0 ** -23 * (v + np.abs(factor * nxt)) + np.abs(nxt) * abs(float(np.float32(factor)) - factor)
    err = np.abs(have - want)
    assert (err <= tol).all(), (factor, float(err.max()), float(tol[np.argmax(err - tol)]))
    return played.sum()


@pytest.mark.parametrize("first_gid", [0, 1])
def test_replay_targets_at_wide_q(first_gid):
    """rezultat_stiha / rezultat_igre for factor 0, 0.1, 1.0 over games played with wide-range q (qmax_hist holds large
    and negative values): seat, T and the -70 pattern exact; the played card within fp32 rounding of the float64 value."""
    n = 8192
    rng = np.random.default_rng(7 + first_gid)
    env, d = _setup(n, 18, first_gid)
    qs, card, qmax, mask = _play(env, d, "wide", 0.1, "plain", rng)
    env.score()
    d["cards"] = card
    L = _lists(d)
    _, _, qmax_ref = _judge_cards(env, d, L, qs, card, qmax, mask, 0.1, first_gid)
    assert np.abs(qmax_ref).max() > 1e30 and (qmax_ref < 0).any()
    for factor in (0.0, 0.1, 1.0):
        assert _targets_check(env, d, L, qmax_ref, factor) > 20 * n
    _, _, rows = env.targets(final_reword_factor=0.1)
    rows = rows.cpu().numpy()
    from oracle import nevronski as N
    for t in range(48):
        on = L["seat"][:, t] != 0xFF
        on &= card[:, t] != 0xFF
        nh = N.history_len(d, t)
        assert (rows[on, t] == (nh + 8 - nh % 8)[on]).all(), t
    env.close()


@pytest.mark.parametrize("mode", [16, 17])
def test_exchange_observation_and_choice_match_restatement(mode):
    """menjaj_talon_v_vektor / menjaj_iz_talona at 65,536 games: observations exact; group and discards for every q
    regime at eps 0 / 0.3 / 1.0 exactly as the restatement (NaN first, -inf a legal value); Q19 hands give no discards."""
    import torch
    from oracle import nevronski as N
    n = 65536
    rng = np.random.default_rng(mode)
    for regime in REGIMES:
        for eps, first_gid in ((0.0, 0), (0.3, 1), (1.0, 2)):
            env, d = _setup(n, mode, first_gid, exchange=False)
            ex = np.nonzero(N.talon_k(d["contract"]) > 0)[0].astype(np.int32)
            if regime == "ties" and eps == 0.0:
                (hand, talon, game), ok = env.obs_exchange(ex)
                assert ok.cpu().numpy().all()
                sub = {k: v[ex] for k, v in d.items()}
                assert (hand.cpu().numpy() == N.unpack(N.hand_dealt(sub["perm"], sub["declarer"]))).all()
                k = N.talon_k(sub["contract"])
                want_t = np.zeros((len(ex), 54, 6), np.float32)
                for j in range(6):
                    want_t[np.arange(len(ex)), sub["perm"][:, 48 + j], j // k] = 1
                assert (talon.cpu().numpy() == want_t).all()
                c = sub["contract"].astype(np.int64)
                want_g = np.zeros((len(ex), 15), np.float32)
                want_g[np.arange(len(ex)), np.where(c <= 3, (c - 1) * 4 + sub["king"], 12 + c - 4)] = 1
                assert (game.cpu().numpy() == want_g).all()
            p = np.concatenate([_q(rng, regime, len(ex), np.zeros(len(ex), np.uint64)),
                                _q(rng, regime, len(ex), np.zeros(len(ex), np.uint64))[:, :6]], axis=1)
            if regime == "nan_one":
                p[np.arange(len(ex)), rng.integers(0, 54, len(ex))] = np.nan
                p[np.arange(len(ex)), 54 + rng.integers(0, 2, len(ex))] = np.nan
            group, disc = env.select_exchange(torch.from_numpy(p), ex, eps)
            group = group.cpu().numpy()
            disc = disc.cpu().numpy().view(np.uint64)
            assert (group[ex] != 0xFF).all(), regime
            sub = {k: v[ex] for k, v in d.items()}
            sub["group"] = group[ex]
            Lx = _lists(sub)
            want_g, want_d = N.choose_exchange(p, sub, Lx, env.seed, ex.astype(np.uint64) + np.uint64(first_gid), eps)
            assert (want_g == group[ex]).all(), (regime, eps)
            assert (want_d == disc[ex]).all(), (regime, eps)
            q19 = Lx["zalozit_n"] < N.talon_k(sub["contract"])
            env.exchange(group, disc)
            assert env.errors() == int(q19.sum()), (regime, eps)
            env.close()


def _masks(x):
    """Device 0/1 fp32 [..., 54] -> int64 bitboards on the host; asserts every entry is 0 or 1."""
    import torch
    assert bool(((x == 0) | (x == 1)).all())
    w = torch.ones(1, dtype=torch.int64, device=x.device) << torch.arange(54, device=x.device)
    return (x.to(torch.int64) * w).sum(-1).cpu().numpy().view(np.uint64)


def _check_obs(o, games, arrs, kind, T, with_mozne=True):
    """Device arrays of one (kind, T) block (reference list order) against the restatement's bitboards for `games`."""
    B = len(games)
    names = {0: ["opp", "hand", "talon"], 1: ["opp", "king", "hand", "talon", "decl", "disc"],
             2: ["opp", "hand", "talon", "decl", "disc"], 3: ["opp", "hand", "decl"]}[kind]
    r = min(T, 48)
    for name, a in zip(names, arrs):
        if name == "opp":
            m = _masks(a).reshape(B, T, 3)
            assert (m[:, :r] == o["opp"][games, :r]).all() and (m[:, r:] == 0).all()
        elif name == "hand":
            m = _masks(a).reshape(B, T)
            assert (m[:, :r] == o["hand"][games, :r]).all() and (m[:, r:] == 0).all()
        elif name == "talon" and kind == 0:
            assert (_masks(a) == o["klop_talon"][games]).all()
        elif name == "talon":
            assert (a.cpu().numpy() == o["talon"][games]).all()
        elif name in ("king", "decl"):
            want = np.zeros((B, 4), np.float32)
            idx = o[name][games]
            want[np.nonzero(idx >= 0)[0], idx[idx >= 0]] = 1
            assert (a.cpu().numpy() == want).all(), name
        elif name == "disc":
            assert (_masks(a) == o["discard"][games]).all()
    if with_mozne:
        assert (_masks(arrs[-1]) == o["mozne"][games]).all()
    assert (o["T"][games] == T).all() and (o["kind"][games] == kind).all()


@pytest.mark.parametrize("mode,first_gid", [(16, 0), (17, 1), (18, 0)])
def test_bucketed_observations_every_play_match_restatement(mode, first_gid):
    """65,536 games through obs_buckets(4) + obs_expand_buckets (the arenas self-play feeds the nets from): at every play,
    every element of every bucket against the restatement; afterwards obs_expand(play=t) for 4,096 games at every t."""
    import torch
    from oracle import nevronski as N
    from tarok_b200.samoigra import _Arena
    n = 65536
    env, d = _setup(n, mode, first_gid)
    ar = _Arena(n, env.torch_device)
    played = np.full((n, 48), 0xFF, np.uint8)
    seen = {"T56": 0, "q19": 0}

    def obs_check(t, sel_dev, cnt):
        total = int(cnt[255])
        env.obs_expand_buckets(total, ar.opp, ar.hand, ar.talon, ar.talon_klop, ar.king, ar.decl, ar.disc)
        d["cards"] = played
        o = N.observation(d, _lists(d), t)
        order = sel_dev[:total].long().cpu().numpy()
        assert (np.sort(order) == np.nonzero(o["live"])[0]).all(), t
        for k in range(127):
            B = int(cnt[k])
            if not B:
                continue
            p, kind, T = k // 28, (k % 28) // 7, 8 * (k % 7 + 1)
            off, row = int(cnt[128 + k]), int(cnt[256 + k])
            games = order[off:off + B]
            assert (((o["seat"][games] + games + first_gid) & 3) == p).all()
            a = ar
            opp = a.opp[row * 162:(row + B * T) * 162].view(B, T, 3, 54)
            hand = a.hand[row * 54:(row + B * T) * 54].view(B, T, 54)
            decl = a.decl[off * 4:(off + B) * 4].view(B, 4)
            talon = a.talon[off * 330:(off + B) * 330].view(B, 6, 55)
            disc = a.disc[off * 54:(off + B) * 54].view(B, 54)
            arrs = {0: [opp, hand, a.talon_klop[off * 54:(off + B) * 54].view(B, 54)],
                    1: [opp, a.king[off * 4:(off + B) * 4].view(B, 4), hand, talon, decl, disc],
                    2: [opp, hand, talon, decl, disc], 3: [opp, hand, decl]}[kind]
            _check_obs(o, games, arrs, kind, T, with_mozne=False)
            seen["T56"] += int(T == 56) * B

    rng = np.random.default_rng(mode)
    # drive with the device's choices (tie-prone q), recording the history the restatement replays
    for t in range(48):
        live = env.live().cpu().numpy()
        if not live.any():
            break
        sel_dev, cnt = env.obs_buckets(4)
        obs_check(t, sel_dev, cnt)
        total = int(cnt[255])
        order = sel_dev[:total].long()
        q = torch.from_numpy(_q(rng, "ties", n, None)).to(env.torch_device)
        q_by_key = {k: q[order[cnt[128 + k]:cnt[128 + k] + cnt[k]]].contiguous() for k in range(127) if cnt[k]}
        cards = torch.full((env.n_alloc,), 0xFF, dtype=torch.uint8, device=env.torch_device)
        env.select_action_buckets(total, q_by_key, [0.0] * 4, cards)
        played[live, t] = cards[:n].cpu().numpy()[live]
        env.step(cards)
    d["cards"] = played
    L = _lists(d)
    # Q19: games whose exchange failed never reach play 0 and expand to ok = 0, zero-filled
    err = np.nonzero((env.meta[:n].cpu().numpy() >> 26) & 1)[0].astype(np.int32)
    if len(err):
        arrs, ok = env.obs_expand(1, 8, err)
        assert not ok.cpu().numpy().any() and all(float(x.abs().sum()) == 0 for x in arrs if x is not None)
    seen["q19"] = len(err)
    sub = np.arange(4096)
    for t in range(48):
        o = N.observation(d, L, t)
        on = o["live"][sub]
        for kind in range(4):
            for T in np.unique(o["T"][sub][on & (o["kind"][sub] == kind)]):
                games = sub[on & (o["kind"][sub] == kind) & (o["T"][sub] == T)].astype(np.int32)
                arrs, ok = env.obs_expand(kind, int(T), games, play=t)
                assert ok.cpu().numpy().all()
                _check_obs(o, games, arrs[:-1], kind, int(T), with_mozne=False)
    assert seen["T56"] > 0
    env.close()


@pytest.mark.parametrize("contract", range(10))
def test_forced_contract_observations_every_play_match_restatement(contract):
    """obs_expand per (kind, T) at every play of 8,192 games of each forced contract (T = 56 in Klop, Solo_brez without
    an exchange entry, Berac early stops), the legal-mask vector included; ragged batch sizes on contract 7."""
    import torch
    from oracle import nevronski as N
    sizes = (8192, 8191, 33, 31, 1) if contract == 7 else (8192,)
    for n in sizes:
        env, d = _setup(n, contract, contract & 1)
        played = np.full((n, 48), 0xFF, np.uint8)
        rng = np.random.default_rng(contract)
        for t in range(48):
            live = env.live().cpu().numpy()
            if not live.any():
                break
            d["cards"] = played
            o = N.observation(d, _lists(d), t)
            assert (o["live"] == live).all(), t
            for kind in range(4):
                for T in np.unique(o["T"][live & (o["kind"] == kind)]):
                    games = np.nonzero(live & (o["kind"] == kind) & (o["T"] == T))[0].astype(np.int32)
                    arrs, ok = env.obs_expand(kind, int(T), games)
                    assert ok.cpu().numpy().all()
                    _check_obs(o, games, arrs, kind, int(T))
            q = torch.from_numpy(_q(rng, "ties", n, None))
            cards, _ = env.select_action(q)
            played[live, t] = cards[:n].cpu().numpy()[live]
            env.step(cards)
        env.close()
