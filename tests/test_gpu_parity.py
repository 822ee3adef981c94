"""GPU parity: the CUDA path, called through the C ABI (tarok_b200.env.TarokEnv -> libtarok_b200.so),
against (a) vectors frozen from the real reference (tests/golden) and (b) the C oracle on the same
seeded inputs.  Bar: bit-exact (all arithmetic on this path is integer)."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN

pytestmark = pytest.mark.gpu

ALL54 = (1 << 54) - 1


def u64(t):
    return t.cpu().numpy().view(np.uint64)


def _env(n, **kw):
    from tarok_b200.env import TarokEnv
    return TarokEnv(n, **kw)


def _meta(env):
    import tarok_b200.env as E
    m = u64(env.meta[: env.n])
    f = lambda sh, b: ((m >> np.uint64(sh)) & np.uint64((1 << b) - 1)).astype(np.int64)
    return dict(contract=f(E.M_CONTRACT, 4), declarer=f(E.M_DECL, 2), king=f(E.M_KING, 3), team=f(E.M_TEAM, 4),
                leader=f(E.M_LEADER, 2), pos=f(E.M_POS, 2), tricks=f(E.M_TRICKS, 4), phase=f(E.M_PHASE, 2),
                err=f(E.M_ERR, 1), group=f(E.M_GROUP, 3), winner=f(E.M_WINNER, 2), trickdone=f(E.M_TRICKDONE, 1),
                plays=f(E.M_PLAYS, 6))


def _replay_on_gpu(g, use_auction=False):
    """Teacher-forces a golden trace set through the stepwise kernels, checking every exposed value."""
    n = len(g["perm"])
    env = _env(n, history=True)
    env.set_deals(g["perm"])
    hands0 = u64(env.hands[:, :n]).T
    if "hands0" in g.files and g["hands0"].any():
        assert (hands0 == g["hands0"]).all()
    if use_auction:
        env.auction(g["intent"])
    else:
        env.force_contract(g["contract"], g["declarer"], g["king"])
    m = _meta(env)
    assert (m["contract"] == g["contract"]).all()
    nk = g["contract"] != 0
    assert (m["declarer"][nk] == g["declarer"][nk]).all()
    assert (m["king"] == g["king"]).all()
    env.exchange(g["group"], g["discard_mask"])
    assert env.errors() == 0
    live = np.ones(n, bool)
    for t in range(48):
        m = _meta(env)
        live = m["phase"] == 2
        assert (live == (g["plays"] > t)).all(), t
        mover = (m["leader"] + m["pos"]) & 3
        assert (mover[live] == g["seat"][live, t]).all(), t
        assert (u64(env.mask[:n])[live] == g["mask"][live, t]).all(), t
        assert (u64(env.legal_mask())[live] == g["mask"][live, t]).all(), t
        env.step(g["card"][:, t])
        if t % 4 == 3:
            m2 = _meta(env)
            assert (m2["trickdone"][live] == 1).all()
            assert (m2["winner"][live] == g["winner"][live, t // 4]).all(), t
    assert env.errors() == 0
    m = _meta(env)
    assert (m["phase"] == 3).all() and (m["plays"] == g["plays"]).all()
    sc = env.score().cpu().numpy()
    assert (sc == g["scores"]).all()
    assert (u64(env.hands[:, :n]).T == g["hands"]).all()
    assert (u64(env.piles[:, :n]).T == g["piles"]).all()
    # conservation: hands, piles and talon partition the deck
    tot = np.bitwise_or.reduce(u64(env.hands[:, :n]), axis=0) | np.bitwise_or.reduce(u64(env.piles[:, :n]), axis=0) \
        | u64(env.talon[:n])
    assert (tot == np.uint64(ALL54)).all()
    hist = env.hist[:, :n].cpu().numpy().T
    played = g["card"] != 0xFF
    assert ((hist & 63)[played] == g["card"][played]).all()
    assert ((hist >> 6)[played] == g["seat"][played]).all()
    assert (hist[~played] == 0xFF).all()
    st = env.stats()
    assert st[18] == n and st[19] == g["plays"].astype(np.int64).sum() and st[20] == 0
    assert (st[0:4] == g["scores"].astype(np.int64).sum(axis=0)).all()
    assert (st[8:18] == np.bincount(g["contract"], minlength=10)).all()
    env.close()


def test_golden_traces_forced(golden):
    _replay_on_gpu(golden("traces_forced.npz"))


def test_golden_traces_full_auction(golden):
    _replay_on_gpu(golden("traces_full.npz"), use_auction=True)


def test_kat_table_scores_and_history_hash():
    rows = json.load(open(os.path.join(GOLDEN, "kat.json")))
    n = len(rows)
    env = _env(n, history=True)
    perm = np.array([r["perm"] for r in rows], np.uint8)
    env.set_deals(perm)
    env.force_contract([r["contract"] for r in rows], [r["declarer"] for r in rows], [r["king"] for r in rows])
    env.exchange([r["group"] for r in rows], np.array([r["discard_mask"] for r in rows], np.uint64))
    cards = np.full((n, 48), 0xFF, np.uint8)
    for i, r in enumerate(rows):
        cards[i, :len(r["cards"])] = r["cards"]
    for t in range(48):
        env.step(cards[:, t])
    sc = env.score().cpu().numpy()
    hist = env.hist[:, :n].cpu().numpy().T
    for i, r in enumerate(rows):
        assert sc[i].tolist() == r["scores"], r
        b = bytearray()
        for t in range(r["plays"]):
            b += bytes((hist[i, t] >> 6, hist[i, t] & 63))
            if r["contract"] == 0 and t % 4 == 3 and t // 4 < 6:      # Klop talon card, seat 9 (SURVEY A.6)
                b += bytes((9, perm[i, 53 - t // 4]))
        assert hashlib.sha256(bytes(b)).hexdigest()[:16] == r["hash"], r
    env.close()


TIP_TO_INDEX = {-1: 0, 0: 19, 1: 1, 2: 5, 3: 9, 4: 13, 5: 14, 6: 15, 7: 16, 8: 17, 9: 18}


def test_auction_fixed_exhaustive(golden):
    a = golden("auction_fixed.npz")
    n = len(a["intents"])
    env = _env(n)
    env.deal()
    idx = np.vectorize(TIP_TO_INDEX.get)(a["intents"]).astype(np.uint8)
    env.auction(idx)
    m = _meta(env)
    assert (m["contract"] == a["contract"]).all()
    nk = a["contract"] != 0
    assert (m["declarer"][nk] == a["declarer"][nk]).all()
    env.close()


def test_deal_matches_oracle_and_is_shard_invariant(oracle):
    n = 30001
    env = _env(n, seed=1234)
    env.deal(first_game_id=0)
    p = env.export_perm().cpu().numpy()
    assert (p == oracle.deal(1234, 0, n)).all()
    env.deal(first_game_id=777)
    assert (env.export_perm().cpu().numpy() == oracle.deal(1234, 777, n)).all()
    # round trip: injecting the exported deal reproduces the state
    h = u64(env.hands).copy(); t = u64(env.talon).copy(); o = u64(env.talon_order).copy()
    env.set_deals(env.export_perm())
    assert (u64(env.hands) == h).all() and (u64(env.talon) == t).all() and (u64(env.talon_order) == o).all()
    env.close()


@pytest.mark.parametrize("gid0", [123456789, 2 ** 33 + 1000])      # odd / even: the Philox game-pair sharing depends on parity
@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 16, 17, 18])
def test_rollout_matches_oracle(oracle, mode, gid0):
    """Whole deals with the Philox players: stepwise kernels == fused kernel == C oracle."""
    n, seed = 20011, 4242
    ref = oracle.rollout(seed, gid0, n, mode)
    env = _env(n, seed=seed, history=True)
    env.rollout(mode, first_game_id=gid0, fused=False)
    m = _meta(env)
    ok = ref["err"] == 0
    assert (m["err"] == ref["err"]).all()
    assert (m["contract"][ok] == ref["contract"][ok]).all()
    nk = ok & (ref["contract"] != 0)
    assert (m["declarer"][nk] == ref["declarer"][nk]).all()
    assert (m["king"][ok] == ref["king"][ok]).all()
    assert (m["plays"] == ref["plays"]).all()
    hist = env.hist[:, :n].cpu().numpy().T
    played = ref["cards"] != 0xFF
    assert ((hist & 63)[played] == ref["cards"][played]).all()
    assert (hist[~played] == 0xFF).all()
    sc = env.scores[:n].cpu().numpy()
    assert (sc == ref["scores"]).all()
    st = env.stats()
    assert (st[0:4] == ref["stats"][0:4]).all() and (st[4:8] == ref["stats"][4:8]).all()
    assert st[19] == ref["stats"][8] and st[20] == ref["stats"][9] and st[18] == ok.sum()
    assert (st[8:18] == np.bincount(ref["contract"][ok], minlength=10)).all()
    state = {k: u64(getattr(env, k)).copy() for k in ("hands", "piles", "talon", "talon_order", "meta")}
    # fused kernel: identical state, scores and statistics
    env.reset_stats()
    env.rollout(mode, first_game_id=gid0, fused=True)
    for k, v in state.items():
        assert (u64(getattr(env, k)) == v).all(), k
    assert (env.scores[:n].cpu().numpy() == sc).all()
    assert (env.stats()[:21] == st[:21]).all()
    assert (env.hist[:, :n].cpu().numpy().T == hist).all()
    env.close()


@pytest.mark.parametrize("mode", [16, 17, 0])
def test_fused_rollout_writes_the_replay_inputs(mode):
    """On a FRESH history-keeping environment the fused rollout must leave everything the replay kernels read -- hands as
    dealt, the declarer's discards, the discard points -- exactly as the stepwise pipeline does (round-1 advisor finding:
    the fused kernel used to leave hands0 / discard stale)."""
    n, seed, gid0 = 30011, 31337, 9
    a, b = _env(n, seed=seed, history=True), _env(n, seed=seed, history=True)
    a.rollout(mode, first_game_id=gid0, fused=False)
    b.rollout(mode, first_game_id=gid0, fused=True)
    for f in ("hands0", "discard", "hands", "piles", "talon", "meta"):
        assert (u64(getattr(a, f)) == u64(getattr(b, f))).all(), f
    assert (a.hist[:, :n].cpu().numpy() == b.hist[:, :n].cpu().numpy()).all()
    da, sa, ra = a.targets()
    db, sb, rb = b.targets()
    assert (sa.cpu().numpy() == sb.cpu().numpy()).all() and (ra.cpu().numpy() == rb.cpu().numpy()).all()
    assert (da.cpu().numpy() == db.cpu().numpy()).all()
    # scoring again (idempotent) from the state the fused kernel wrote
    sc = b.scores[:n].cpu().numpy().copy()
    b.reset_stats()
    assert (b.score().cpu().numpy() == sc).all()
    a.close(); b.close()


@pytest.mark.parametrize("mode", [17, 16, 0])
def test_chain_of_random_steps_with_lazy_masks_leaves_the_same_state(mode):
    """A chain of in-kernel random steps writes the legal masks in its last launch only (TAROK_OPT_LAZY_MASK, default on):
    after every chain -- whatever its length, also with games finishing inside it (Berac early stops in mode 17) and with
    warps that fall back to the general path -- masks, meta, hands and the trick-derived scores equal those of a run
    whose every launch writes its masks."""
    import tarok_b200.env as E
    n, seed, gid0 = 50021, 2718, 3
    a, b = _env(n, seed=seed), _env(n, seed=seed)
    b.set_lazy_mask(False)
    a.deal(gid0); b.deal(gid0)
    if mode == 17:
        a.auction_synth(17); b.auction_synth(17)
        a.step_random(2); b.step_random(2)                       # the contracts without an exchange run ahead: general path later
        a.exchange_synth(True); b.exchange_synth(True)
    else:
        a.force_contract_synth(mode); b.force_contract_synth(mode)
        a.exchange_synth(False); b.exchange_synth(False)
    for chunk in (1, 2, 5, 3, 13, 1, 30):
        a.step_random(chunk); b.step_random(chunk)
        for f in ("mask", "meta", "hand_slots"):
            assert (u64(getattr(a, f)) == u64(getattr(b, f))).all(), (f, chunk)
        assert (u64(a.legal_mask()) == u64(a.mask[:n])).all()    # and they are the masks of the state
    assert (a.score().cpu().numpy() == b.score().cpu().numpy()).all()
    assert (a.stats()[:21] == b.stats()[:21]).all()
    a.close(); b.close()


@pytest.mark.parametrize("gid0,rows", [(6, 3), (6, 2), (7, 3), (6, 0)])
def test_draw_cache_never_changes_a_draw(gid0, rows):
    """The position-0 launch of a trick leaves the pair's random lanes of positions 1-3 behind for the next three launches
    (the draw cache).  Whatever the interleaving -- the opening card supplied from outside (nothing cached for that trick: the
    entry carries the previous trick's tag), a supplied card in the middle of a cached trick, single launches and chains,
    the same handle re-dealt under another first game id (another epoch) and back -- every in-kernel draw must be the one a
    plain random rollout makes, because a draw depends on (seed, game id, play index) only."""
    import torch
    n, seed = 30011, 99
    a = _env(n, seed=seed, history=True)
    a.rollout(16, first_game_id=gid0, fused=False)
    want = a.hist[:, :n].clone()                                  # [48, n] seat << 6 | card
    want_scores = a.scores[:n].cpu().numpy().copy()
    b = _env(n, seed=seed, history=True)
    b.set_draw_cache(rows)                                        # positions 1..rows read the cache (a is on the default, 3)
    b.rollout(16, first_game_id=gid0 + 2 * n, fused=False)        # fills the cache under another epoch and other game ids
    b.deal(gid0)
    b.force_contract_synth(16)
    b.exchange_synth(False)
    supplied = {0, 5, 10, 15, 16, 17, 18, 19, 24, 30, 33, 44}
    t = 0
    while t < 48:
        if t in supplied:
            b.step((want[t] & 63).contiguous())
            t += 1
        else:
            run = 1
            while t + run < 48 and (t + run) not in supplied and run < 3 + (t % 5):
                run += 1
            b.step_random(run)
            t += run
        assert (b.hist[:t, :n] == want[:t]).all(), t
    assert (b.score().cpu().numpy() == want_scores).all()
    # back to the first handle: same ids again (a new epoch on a cache holding the same blocks), chained
    a.reset_stats()
    a.rollout(16, first_game_id=gid0, fused=False)
    assert (a.hist[:, :n] == want).all() and (a.scores[:n].cpu().numpy() == want_scores).all()
    a.close(); b.close()


def test_desynchronised_batch_takes_the_general_path(oracle):
    """Games that start playing at different times (here: the contracts without a talon exchange play three cards before
    the others have exchanged) break the lock-step hint inside most warps; the per-warp vote must then send them through
    the general path, with the same games as a result (the Philox draws depend on the game and its own play index only)."""
    import tarok_b200.env as E
    n, seed, gid0 = 40001, 777, 5
    ref = oracle.rollout(seed, gid0, n, E.MODE_AUCTION_UNIFORM)
    env = _env(n, seed=seed, history=True)
    env.deal(gid0)
    env.auction_synth(E.MODE_AUCTION_UNIFORM)
    waiting = (_meta(env)["phase"] == E.PH_EXCHANGE)
    assert 0.05 < waiting.mean() < 0.95                      # a real mix inside every warp
    env.step_random(3)                                       # only Klop / Berac / Solo_brez games move
    m = _meta(env)
    assert (m["plays"][waiting] == 0).all() and (m["plays"][~waiting & (ref["err"] == 0)] == 3).all()
    env.exchange_synth(True)
    env.step_random(48)                                      # 45 more for the early starters, 48 for the rest
    sc = env.score().cpu().numpy()
    assert (sc == ref["scores"]).all()
    assert (_meta(env)["plays"] == ref["plays"]).all()
    hist = env.hist[:, :n].cpu().numpy().T
    played = ref["cards"] != 0xFF
    assert ((hist & 63)[played] == ref["cards"][played]).all()
    st = env.stats()
    assert (st[0:8] == ref["stats"][0:8]).all() and st[19] == ref["stats"][8] and st[20] == ref["stats"][9]
    env.close()


def test_fused_setup_equals_separate_kernels():
    import tarok_b200.env as E
    n = 70001
    for mode in (16, 17, 18, 0, 7, 8):
        a, b = _env(n, seed=99, history=True), _env(n, seed=99, history=True)
        a.setup_synth(mode, 555)
        b.deal(555)
        b.auction_synth(mode) if mode in (17, 18) else b.force_contract_synth(mode)
        b.exchange_synth(mode == E.MODE_AUCTION_UNIFORM)
        for f in ("hands", "piles", "talon", "talon_order", "meta", "mask", "hands0", "discard"):
            assert (u64(getattr(a, f)) == u64(getattr(b, f))).all(), (mode, f)
        assert a.stats()[21] == b.stats()[21]
        a.close(); b.close()


def test_teacher_forced_replay_at_full_size(oracle):
    """BASELINE config 2 size: 1,048,576 Navadna deals played on the GPU, then EVERY game replayed
    card by card through the C oracle (legality, trick winners, scores)."""
    import tarok_b200.env as E
    n = 1 << 20
    env = _env(n, seed=7, history=True)
    env.deal(0)
    perm = env.export_perm().cpu().numpy()
    env.force_contract_synth(E.MODE_NAVADNA_MIX)
    env.exchange_synth(False)
    m = _meta(env)
    disc = u64(env.discard[:n]).copy()
    for _ in range(48):
        env.step_random()
    sc = env.score().cpu().numpy()
    hist = env.hist[:, :n].cpu().numpy().T
    cards = np.where(hist == 0xFF, 0xFF, hist & 63).astype(np.uint8)
    rep = oracle.replay(perm, m["contract"].astype(np.uint8), m["declarer"].astype(np.uint8),
                        m["king"].astype(np.uint8), m["group"].astype(np.uint8), disc, cards, want_state=False)
    gerr = _meta(env)["err"]
    ok = gerr == 0
    assert ok.mean() > 0.999
    assert (rep["err"][ok] == 0).all()
    assert (rep["scores"][ok] == sc[ok]).all()
    assert ((hist >> 6)[ok] == rep["seat"][ok]).all()
    # size-independent properties
    assert (u64(env.hands[:, :n])[:, ok] == 0).all()
    tot = np.bitwise_or.reduce(u64(env.piles[:, :n]), axis=0) | u64(env.talon[:n])
    assert (tot[ok] == np.uint64(ALL54)).all()
    st = env.stats()
    assert st[19] == 48 * ok.sum() and st[18] == ok.sum()
    env.close()


def test_illegal_action_sets_error_bit_and_stops_the_game():
    n = 1024
    env = _env(n, seed=3)
    env.deal()
    env.force_contract_synth(0)
    mask = u64(env.mask[:n])
    legal_lowest = np.array([int(x & -x).bit_length() - 1 for x in mask.astype(object)], np.uint8)
    cards = legal_lowest.copy()
    bad = np.arange(n) % 7 == 0
    hands0 = u64(env.hands[0, :n])
    for i in np.nonzero(bad)[0]:   # a card the leader does not hold
        cards[i] = next(c for c in range(54) if not (int(hands0[i]) >> c) & 1)
    env.step(cards)
    m = _meta(env)
    assert (m["err"] == bad).all()
    assert (m["phase"][bad] == 3).all() and (m["phase"][~bad] == 2).all()
    assert env.stats()[21] == bad.sum()
    assert (u64(env.hands[0, :n])[bad] == hands0[bad]).all()      # state untouched
    # the survivors play on; at the trick-closing position (the launch that re-seats the hand slots) some of them send a
    # card they do not hold and some an id that is no card at all
    def lowest_legal():
        mk = u64(env.mask[:n])
        return np.array([max(int(x & -x).bit_length() - 1, 0) for x in mk.astype(object)], np.uint8)
    env.step(lowest_legal())
    env.step(lowest_legal())
    cards = lowest_legal()
    before = u64(env.hands[:, :n]).copy()
    live = ~bad
    bad2 = live & (np.arange(n) % 5 == 0)
    bad3 = live & ~bad2 & (np.arange(n) % 11 == 0)
    mover = (_meta(env)["leader"] + _meta(env)["pos"]) & 3
    for i in np.nonzero(bad2)[0]:
        cards[i] = next(c for c in range(54) if not (int(before[mover[i], i]) >> c) & 1)
    cards[bad3] = 200
    env.step(cards)
    m = _meta(env)
    assert (m["err"] == (bad | bad2 | bad3)).all()
    assert (m["tricks"][live & ~bad2 & ~bad3] == 1).all() and (m["tricks"][bad2 | bad3] == 0).all()
    after = u64(env.hands[:, :n])
    assert (after[:, bad2 | bad3] == before[:, bad2 | bad3]).all()          # refused: nothing moved, nothing re-seated
    assert env.stats()[21] == bad.sum() + bad2.sum() + bad3.sum()
    ok = live & ~bad2 & ~bad3
    assert ((np.bitwise_count(before[:, ok]).sum(axis=0) - np.bitwise_count(after[:, ok]).sum(axis=0)) == 1).all()
    env.close()


def test_invalid_exchange_is_an_error():
    n = 512
    env = _env(n, seed=5)
    env.deal()
    env.force_contract(np.full(n, 1, np.uint8), np.zeros(n, np.uint8), np.zeros(n, np.uint8))
    disc = np.zeros(n, np.uint64)
    hands = u64(env.hands[0, :n])
    kings = np.uint64((1 << 7) | (1 << 15) | (1 << 23) | (1 << 31))
    disc[:] = hands & kings          # kings can never be laid down (Q8); also wrong count
    env.exchange(np.zeros(n, np.uint8), disc)
    assert (_meta(env)["err"] == 1).all()
    env.close()


def test_host_buffer_entry_matches_device_path(oracle):
    import torch
    n = 50000
    ref = oracle.rollout(11, 0, n, 16)
    for fused in (False, True):
        env = _env(n, seed=11)
        scores = torch.empty((n, 4), dtype=torch.int16).pin_memory()
        stats = torch.zeros(32, dtype=torch.int64).pin_memory()
        env.rollout_host(ref["perm"], ref["contract"], ref["declarer"], ref["king"], scores, stats, fused=fused)
        torch.cuda.synchronize()
        assert (scores.numpy() == ref["scores"]).all()
        assert stats[19] == ref["stats"][8]
        assert (stats[0:8].numpy() == ref["stats"][0:8]).all()
        env.close()


@pytest.mark.parametrize("mode", [0, 16, 17])
def test_deal_records_match_permutation_rows(oracle, mode):
    """20-byte deal records carry the same deal (incl. the ORDER of the talon, which Klop consumes card by card) and the same
    forced contract as the 57-byte row format: identical scores, and both agree with the oracle."""
    import torch
    from tarok_b200.env import pack_records
    n = 300001                                                       # ragged: not a multiple of the chunk or the CTA
    ref = oracle.rollout(77, 0, n, mode)
    rec, bad = pack_records(ref["perm"], ref["contract"], ref["declarer"], ref["king"])
    assert bad == 0 and rec.shape == (n, 20)
    out = []
    for records in (False, True):
        env = _env(n, seed=77)
        scores = torch.empty((n, 4), dtype=torch.int16).pin_memory()
        stats = torch.zeros(32, dtype=torch.int64).pin_memory()
        if records:
            env.rollout_records(rec, scores, stats)
        else:
            env.rollout_host(ref["perm"], ref["contract"], ref["declarer"], ref["king"], scores, stats, fused=True)
        torch.cuda.synchronize()
        out.append((scores.numpy().copy(), stats.numpy().copy()))
        env.close()
    assert (out[0][0] == out[1][0]).all() and (out[0][1] == out[1][1]).all()
    if mode != 17:        # the host entries always take talon group 0 (Bot_igralec, Igralec.py:162); mode 17 of the oracle draws it
        assert (out[1][0] == ref["scores"]).all()
        assert out[1][1][19] == ref["stats"][8] and (out[1][1][0:8] == ref["stats"][0:8]).all()
    else:
        assert len(set(ref["contract"].tolist())) >= 9          # every contract family went through both formats


def test_deal_records_reject_what_the_rows_reject():
    """Rows that are not permutations / out-of-range contracts become error games in both formats."""
    import torch
    from tarok_b200.env import pack_records
    n = 4096
    rng = np.random.default_rng(5)
    perm = np.stack([rng.permutation(54) for _ in range(n)]).astype(np.uint8)
    contract = np.full(n, 3, np.uint8); declarer = (np.arange(n) % 4).astype(np.uint8); king = (np.arange(n) % 4).astype(np.uint8)
    perm[10, 5] = perm[10, 6]                    # duplicate card in seat 0 (the missing card would default to seat 0)
    perm[11, 50] = 54                            # out-of-range id in the talon
    contract[12] = 11                            # no such contract
    declarer[13] = 4
    king[14] = 5                                 # king game with no valid suit
    rec, bad = pack_records(perm, contract, declarer, king)
    assert bad == 3                              # rows 10, 11, 13; rows 12 and 14 are well-formed records of an invalid call
    out = {}
    for name in ("rows", "records"):
        env = _env(n, seed=1)
        scores = torch.empty((n, 4), dtype=torch.int16).pin_memory()
        stats = torch.zeros(32, dtype=torch.int64).pin_memory()
        if name == "rows":
            env.rollout_host(perm, contract, declarer, king, scores, stats, fused=True)
        else:
            env.rollout_records(rec, scores, stats)
        torch.cuda.synchronize()
        out[name] = (scores.numpy().copy(), stats.numpy().copy())
        env.close()
    assert (out["rows"][0] == out["records"][0]).all()
    assert (out["rows"][1] == out["records"][1]).all()
    assert out["rows"][1][20] == 5 and out["rows"][1][18] == n - 5          # error games / finished games
    assert (out["rows"][0][10:15] == 0).all()


def test_no_cpu_fallback_symbols_loaded():
    """The product path is the CUDA library: it must be loaded in-process and have launched kernels."""
    env = _env(1000)
    before = env.launches
    env.rollout(0)
    assert env.launches - before == 51          # one graph replay: the hand-over kernel + setup + 48 x play_step + score
    env.set_graph(False)
    before = env.launches
    env.rollout(0)
    assert env.launches - before == 50          # plain launches: setup + 48 x play_step + score
    with open("/proc/self/maps") as f:
        assert "libtarok_b200.so" in f.read()
    env.close()


@pytest.mark.parametrize("n", [1, 2, 3, 511, 512, 513, 1025])
def test_ragged_batch_sizes(oracle, n):
    """Batches that do not fill the 512-game tile (incl. a single game) match the oracle."""
    for mode in (16, 18):
        ref = oracle.rollout(5, 40, n, mode)
        env = _env(n, seed=5, history=True)
        env.rollout(mode, first_game_id=40)
        assert (env.scores[:n].cpu().numpy() == ref["scores"]).all()
        hist = env.hist[:, :n].cpu().numpy().T
        played = ref["cards"] != 0xFF
        assert ((hist & 63)[played] == ref["cards"][played]).all()
        st = env.stats()
        assert st[19] == ref["stats"][8] and st[18] + st[20] == n
        env.close()


def _force_graph(env):
    """TAROK_OPT_GRAPH = 2: the stepwise rollout replays its CUDA graph at every batch size (set_graph passes 0 or 1)."""
    env._check(env._lib.tarok_set_option(env._h, 8, 2))


def _score_windows(env, ref, windows, what):
    for a, b in windows:
        sc = env.scores[a:b].cpu().numpy()
        bad = np.flatnonzero((sc != ref["scores"][a:b]).any(axis=1))
        assert bad.size == 0, "%s: games %s of [%d, %d) differ from the oracle" % (what, (a + bad[:8]).tolist(), a, b)


def test_config5_size_properties(oracle):
    """16,777,216 concurrent deals (BASELINE config 5 total) with bidding: see _large_batch_against_oracle."""
    _large_batch_against_oracle(oracle, 1 << 24, (17,))


def test_config3_size_matches_oracle(oracle):
    """4,194,304 concurrent deals (BASELINE config 3 at N = 1), uniform and Bot-model bids: see _large_batch_against_oracle."""
    _large_batch_against_oracle(oracle, 1 << 22, (17, 18))


def _large_batch_against_oracle(oracle, n, modes):
    """Size-independent invariants, then bench.py's sequence for batch 1 of the leg against the oracle over every game.
    Above 3 M deals the defaults change (no CUDA graph, no draw cache): the statistics and three windows of scores must also
    hold with the draw cache forced on, through the fused kernel and through the stepwise rollout with the graph forced."""
    import tarok_b200.env as E
    env = _env(n, seed=2026)
    env.rollout(E.MODE_AUCTION_UNIFORM, first_game_id=0)
    st = env.stats()
    assert st[18] + st[20] == n                                   # every deal finished or was flagged
    assert st[8:18].sum() == st[18] and st[20] < n // 10000
    assert (st[0:4].sum() == st[4:8].sum())                        # seat sums and player sums are the same total
    import torch
    hands = env.hands[:, :n]
    meta = env.meta[:n]
    err = ((meta >> E.M_ERR) & 1).bool()
    berac = (((meta & 15) == 7) | ((meta & 15) == 9))
    assert bool(((hands != 0).any(dim=0) <= (berac | err)).all())  # only Berac (early stop) leaves cards in hand
    allc = env.piles[0, :n] | env.piles[1, :n] | env.piles[2, :n] | env.piles[3, :n] | env.talon[:n] \
        | hands[0] | hands[1] | hands[2] | hands[3]
    assert bool((allc == ALL54).all())                              # hands, piles and talon partition the deck
    plays = (meta >> E.M_PLAYS) & 63
    assert int(plays.sum().item()) == st[19]
    # fused kernel reproduces the statistics at this size
    env.reset_stats()
    env.rollout(E.MODE_AUCTION_UNIFORM, first_game_id=0, fused=True)
    assert (env.stats()[:21] == st[:21]).all()
    del hands, meta, err, berac, allc, plays        # zero-copy views must be dropped before the handle can be destroyed

    gid0 = n                                        # bench.py's batch 1 of the leg: global game ids [total, 2 * total)
    mid = 1 << 23 if n > 1 << 23 else n // 2
    windows = [(0, 20000), (mid - 10000, mid + 10000), (n - 20000, n)]
    env.set_materialise(False)
    for mode in modes:
        ref = oracle.rollout(2026, gid0, n, mode, full=False)
        want = oracle.device_stats(ref)
        for how in ("bench", "draw cache 3", "fused", "stepwise, graph forced"):
            env.reset_stats()
            if how == "fused":
                env.rollout(mode, first_game_id=gid0, fused=True)
            elif how.startswith("stepwise"):
                _force_graph(env)
                env.rollout(mode, first_game_id=gid0, fused=False)
                env.set_graph(True)
            else:
                env.set_draw_cache(3 if how == "draw cache 3" else -1)
                env.setup_synth(mode, gid0)
                env.step_random(48)
                env.score()
            st = env.stats()[:21]
            what = "mode %d, %s" % (mode, how)
            assert (st == want).all(), "%s: stats %s != oracle %s" % (what, st.tolist(), want.tolist())
            _score_windows(env, ref, windows, what)
        env.set_draw_cache(-1)
        del ref
    env.close()


def test_near_maximum_batch_uses_64_bit_indices(oracle):
    """400 M concurrent deals (61 GB of state; the handle takes up to 2^29): row offsets into the 12-row trick log and the
    48-row history exceed 2^32 there.  Stepwise (trick log -> k_score) and fused (registers) must still agree, and the
    stepwise scores of the last 100,000 games and of 100,000 games around game 2^28 must be the oracle's."""
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < 90 << 30:
        pytest.skip("needs 90 GB of free device memory")
    n = 400_000_000
    env = _env(n, seed=7)
    env.set_materialise(False)
    env.rollout(17, first_game_id=0, fused=False)
    a = env.stats().copy()
    for lo in ((1 << 28) - 50_000, n - 100_000):
        ref = oracle.rollout(7, lo, 100_000, 17, full=False)
        sc = env.scores[lo:lo + 100_000].cpu().numpy()
        assert (sc == ref["scores"]).all(), lo
    env.reset_stats()
    env.rollout(17, first_game_id=0, fused=True)
    b = env.stats().copy()
    env.close()
    assert (a[:21] == b[:21]).all()
    assert a[18] + a[20] == n and a[20] < n // 10000


def test_history_past_32_bit_row_offsets(oracle):
    """100,000,000 history-keeping deals: the [48, n] history rows start past 2^32 bytes from play 43 on (48 x n_alloc > 2^32
    above about 91.4 M deals), so every row offset must be 64-bit.  The history, the hands as dealt and the discards of the
    first and last 50,000 games are the oracle's, through the stepwise and the fused rollout; a 50,000-game handle that holds
    the last games under the same ids gives the same replay targets and observations."""
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < 55 << 30:
        pytest.skip("needs 55 GB of free device memory")
    n, w, gid0, seed, mode = 100_000_000, 50_000, 2 ** 32 + 4321, 99, 16
    assert 47 * (n + 512) > 1 << 32
    env = _env(n, seed=seed, history=True)
    refs = {lo: oracle.rollout(seed, gid0 + lo, w, mode) for lo in (0, n - w)}
    for fused in (False, True):
        env.rollout(mode, first_game_id=gid0, fused=fused)
        for lo, ref in refs.items():
            what = "%s rollout, games [%d, %d)" % ("fused" if fused else "stepwise", lo, lo + w)
            rep = oracle.replay(ref["perm"], ref["contract"], ref["declarer"], ref["king"], ref["group"], ref["discard"],
                                ref["cards"], want_state=False)
            hist = env.hist[:, lo:lo + w].cpu().numpy().T
            want = np.where(ref["cards"] == 0xFF, 0xFF, (rep["seat"] << 6) | ref["cards"]).astype(np.uint8)
            assert (hist == want).all(), what
            hands0 = u64(env.hands0[:, lo:lo + w])
            for s in range(4):
                bits = np.uint64(1) << ref["perm"][:, 12 * s:12 * s + 12].astype(np.uint64)
                assert (hands0[s] == np.bitwise_or.reduce(bits, axis=1)).all(), (what, s)
            assert (u64(env.discard[lo:lo + w]) == ref["discard"]).all(), what
            assert (env.scores[lo:lo + w].cpu().numpy() == ref["scores"]).all(), what

    small = _env(w, seed=seed, history=True)
    small.rollout(mode, first_game_id=gid0 + n - w, fused=True)
    sel = np.arange(n - w, n, dtype=np.int32)
    big_t, small_t = env.targets(sel), small.targets()
    for x, y in zip(big_t, small_t):
        assert (x.cpu().numpy() == y.cpu().numpy()).all()
    seat, rows = small_t[1].cpu().numpy(), small_t[2].cpu().numpy()
    sub = np.arange(4096)
    for t in (0, 21, 47):
        played = seat[sub, t] != 0xFF                  # the observation a replay sample of play t was made from: (type, T)
        for T in np.unique(rows[sub, t][played]):
            games = sub[played & (rows[sub, t] == T)].astype(np.int32)
            a, ok_a = env.obs_expand(1, int(T), games + (n - w), play=t)
            b, ok_b = small.obs_expand(1, int(T), games, play=t)
            assert ok_b.cpu().numpy().all() and (ok_a.cpu().numpy() == ok_b.cpu().numpy()).all(), (t, T)
            for x, y in zip(a, b):
                assert (x.cpu().numpy() == y.cpu().numpy()).all(), (t, T)
    del big_t, small_t
    small.close()
    env.close()


@pytest.mark.parametrize("mode", [0, 7, 9, 16, 17, 18])
def test_scores_only_path_matches_oracle(oracle, mode):
    """tarok_score without pile materialisation (TAROK_OPT_MATERIALISE = 0): same scores and statistics."""
    n, seed = 30001, 808
    ref = oracle.rollout(seed, 64, n, mode, full=False)
    env = _env(n, seed=seed)
    env.set_materialise(False)
    env.rollout(mode, first_game_id=64)
    assert (env.scores[:n].cpu().numpy() == ref["scores"]).all()
    st = env.stats()
    assert (st[0:8] == ref["stats"][0:8]).all() and st[19] == ref["stats"][8]
    env.close()


@pytest.mark.parametrize("impl,pdl,lock", [(1, False, False), (1, True, False), (1, False, True), (2, True, False), (2, False, False),
                                           (3, True, True), (3, False, True)])
def test_every_play_step_variant_matches_oracle(oracle, impl, pdl, lock):
    """The selectable play_step implementations (plain / TMA-staged general path / persistent prefetching lock-step kernel, PDL
    on/off, lock-step specialisation on/off) all produce the oracle's games, graph-backed or not."""
    n, seed = 70001, 31
    for mode in (17, 0):
        ref = oracle.rollout(seed, 10, n, mode)
        env = _env(n, seed=seed, history=True)
        env.set_step_impl(impl); env.set_pdl(pdl); env.set_lockstep(lock)
        env.rollout(mode, first_game_id=10)
        assert (env.scores[:n].cpu().numpy() == ref["scores"]).all()
        hist = env.hist[:, :n].cpu().numpy().T
        played = ref["cards"] != 0xFF
        assert ((hist & 63)[played] == ref["cards"][played]).all()
        # externally supplied actions through the same variant: replay the oracle's cards
        env.setup_synth(mode, 10)
        for t in range(48):
            env.step(ref["cards"][:, t])
        assert (env.score().cpu().numpy() == ref["scores"]).all() and env.errors() == int(ref["err"].sum())
        env.close()


@pytest.mark.parametrize("lock", [True, False])
def test_hand_slots_follow_the_trick_leader(lock):
    """TAROK_F_HANDS is kept in leader-relative slots (row j = seat (leader + j) & 3): check the invariant against the
    seat-indexed copy at every play of a mixed-contract batch (Berac: the declarer leads from the start), with the lock-step
    kernels and with the general path, and that the legal mask is cut from the mover's hand (= row `pos`)."""
    import torch
    import tarok_b200.env as E
    n = 20000
    env = _env(n, seed=99)
    env.set_lockstep(lock)
    env.setup_synth(E.MODE_AUCTION_UNIFORM, 0)
    idx = torch.arange(n, device="cuda")
    for t in range(48):
        meta = env.meta[:n]
        leader = (meta >> E.M_LEADER) & 3
        pos = (meta >> E.M_POS) & 3
        live = ((meta >> E.M_PHASE) & 3) == E.PH_PLAY
        seats = env.hands[:, :n]
        slots = env.hand_slots[:, :n]
        for j in range(4):
            assert bool((slots[j] == seats[(leader + j) & 3, idx]).all()), (t, j)
        mask = env.mask[:n]
        assert bool(((mask & ~slots[pos, idx]) == 0)[live].all()), t
        assert bool((mask[live] != 0).all()) and bool((mask[~live] == 0).all()), t
        del meta, slots, mask
        env.step_random(1)
    env.close()


def test_graph_backed_rollout_equals_plain_launches():
    """tarok_rollout_stepwise replays a captured CUDA graph whose kernels read first_gid and the draw-cache epoch from device
    memory (TAROK_OPT_GRAPH, default on).  Replays under different game ids (odd and even: the draw cache is bypassed for
    odd ids), modes and after option changes must equal the plain 50-launch path bit for bit, on any stream."""
    import torch
    n, seed = 30011, 77
    a, b = _env(n, seed=seed, history=True), _env(n, seed=seed, history=True)
    b.set_graph(False)
    side = torch.cuda.Stream()
    for it, (mode, gid0) in enumerate([(16, 0), (16, 4 * n), (17, 4 * n + 1), (16, 2 ** 40 + 6), (0, 7), (16, 0), (18, 12)]):
        a.reset_stats(); b.reset_stats()
        if it == 3:
            a.set_lazy_mask(False); b.set_lazy_mask(False)       # an option change drops the captured graphs
        if it == 4:
            a.set_lazy_mask(True); b.set_lazy_mask(True)
        if it % 2:
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                a.rollout(mode, first_game_id=gid0, fused=False)
            torch.cuda.current_stream().wait_stream(side)
        else:
            a.rollout(mode, first_game_id=gid0, fused=False)
        b.rollout(mode, first_game_id=gid0, fused=False)
        for f in ("hand_slots", "meta", "mask", "talon", "talon_order", "scores"):
            assert (u64(getattr(a, f)) == u64(getattr(b, f))).all(), (it, f)
        assert (a.hist[:, :n] == b.hist[:, :n]).all(), it
        assert (a.stats()[:21] == b.stats()[:21]).all(), it
        assert a.launches - b.launches == it + 1, it             # the 50 kernels of the graph are counted, + the one-thread hand-over kernel
    # two graph-backed handles in flight at once on different streams: each reads its own slot of run parameters
    c = _env(n, seed=seed, history=True)
    a.reset_stats(); b.reset_stats(); c.reset_stats()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        c.rollout(16, first_game_id=10 * n, fused=False)
    a.rollout(16, first_game_id=20 * n, fused=False)
    torch.cuda.current_stream().wait_stream(side)
    b.rollout(16, first_game_id=10 * n, fused=False)
    assert (c.hist[:, :n] == b.hist[:, :n]).all() and (u64(c.scores) == u64(b.scores)).all()
    b.rollout(16, first_game_id=20 * n, fused=False)
    assert (a.hist[:, :n] == b.hist[:, :n]).all() and (u64(a.scores) == u64(b.scores)).all()
    c.close()
    # stepping by hand after a graph-backed rollout starts from a known state
    a.deal(5); b.deal(5)
    a.force_contract_synth(16); b.force_contract_synth(16)
    a.exchange_synth(False); b.exchange_synth(False)
    a.step_random(48); b.step_random(48)
    assert (a.score().cpu().numpy() == b.score().cpu().numpy()).all()
    a.close(); b.close()


def test_reseed_equals_a_fresh_environment():
    """tarok_reseed gives an existing handle a new run seed: every later draw (deal, bids, exchange, plays -- stepwise, graph-backed
    and fused) is the one a handle created with that seed makes, also right after rollouts under the old seed (stale graphs and
    draw-cache entries must not leak through)."""
    n = 20011
    a = _env(n, seed=111, history=True)
    for mode in (16, 18):
        a.rollout(mode, first_game_id=4)                      # old seed: fills the graph cache and the draw cache
    a.reseed(222)
    b = _env(n, seed=222, history=True)
    for mode, fused in ((16, False), (18, False), (16, True)):
        a.reset_stats(); b.reset_stats()
        a.rollout(mode, first_game_id=4, fused=fused); b.rollout(mode, first_game_id=4, fused=fused)
        assert (a.hist[:, :n] == b.hist[:, :n]).all() and (u64(a.scores) == u64(b.scores)).all(), (mode, fused)
        assert (a.stats()[:21] == b.stats()[:21]).all()
    a.close(); b.close()


def test_pipeline_is_cuda_graph_capturable():
    """Every entry point only enqueues stream-ordered work (incl. the programmatic-dependent-launch chain of play_steps), so a
    caller can capture deal -> 48 steps -> score into a CUDA graph and replay it."""
    import torch
    n = 30000
    env = _env(n, seed=5)
    env.rollout(16, first_game_id=0)
    ref, sc_ref = env.stats().copy(), env.scores[:n].clone()
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        env.reset_stats(); env.rollout(16, first_game_id=0)          # warm-up on the capture stream
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=s):
            env.reset_stats()
            env.setup_synth(16, 0)
            env.step_random(48)
            env.score()
    for _ in range(2):
        env.scores.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert (env.stats()[:21] == ref[:21]).all() and bool((env.scores[:n] == sc_ref).all())
    del sc_ref, g
    env.close()


def test_error_paths_are_loud():
    """Bad arguments and bad inputs come back as error codes / error bits with a message, never silently."""
    import torch
    from tarok_b200 import _lib
    from tarok_b200.env import TarokEnv
    with pytest.raises(_lib.TarokLibraryError, match="n_games"):
        TarokEnv(0)
    env = _env(600, history=False)
    with pytest.raises(_lib.TarokLibraryError, match="bad contract mode"):
        env.force_contract_synth(12)
    with pytest.raises(_lib.TarokLibraryError, match="bad auction mode"):
        env.auction_synth(3)
    with pytest.raises(_lib.TarokLibraryError, match="HISTORY"):
        env.view(7)                                              # hist was not requested
    with pytest.raises(ValueError):
        env.set_deals(np.zeros((599, 54), np.uint8))             # wrong shape
    # a deal that is not a permutation of the 54 cards is flagged per game and never played
    perm = np.tile(np.arange(54, dtype=np.uint8), (600, 1))
    perm[7, 3] = perm[7, 4]                                       # duplicate card
    perm[9, 0] = 77                                               # out of range
    env.set_deals(perm)
    env.force_contract_synth(0)
    m = _meta(env)
    assert m["err"].nonzero()[0].tolist() == [7, 9] and (m["phase"][[7, 9]] == 3).all()
    env.step_random(48)
    sc = env.score().cpu().numpy()
    assert (sc[[7, 9]] == 0).all()
    st = env.stats()
    assert st[20] == 2 and st[18] == 598
    # a handle cannot be destroyed under a live zero-copy view
    view = env.meta
    env._views.clear()
    with pytest.raises(_lib.TarokLibraryError, match="exported tensors still alive"):
        env._check(env._lib.tarok_destroy(env._h))
    del view, m
    env.close()


def test_device_randomness_is_uniform():
    """Chi-square checks of the Philox deal / talon order / random-play draws (the oracle shares the generator, so
    parity alone would not reveal a biased one)."""
    import torch
    n = 1 << 21
    env = _env(n, seed=123456789)
    env.deal(0)
    hands = env.hands[:, :n]
    talon = env.talon[:n]
    # 1. every card lands in each hand with probability 12/54 and in the talon with 6/54
    chi = 0.0
    for c in range(54):
        obs = [float(((hands[s] >> c) & 1).sum().item()) for s in range(4)] + [float(((talon >> c) & 1).sum().item())]
        exp = [n * 12 / 54] * 4 + [n * 6 / 54]
        chi += sum((o - e) ** 2 / e for o, e in zip(obs, exp))
    assert chi < 54 * 4 + 6 * (2 * 54 * 4) ** 0.5, chi          # 216 degrees of freedom, ~6 sigma
    # 2. the talon order is a uniform permutation: rank pattern of the six ids -> 720 classes
    order = env.talon_order[:n]
    ids = torch.stack([(order >> (6 * i)) & 63 for i in range(6)], dim=1)
    ranks = ids.argsort(dim=1).argsort(dim=1)
    code = (ranks * torch.tensor([7 ** i for i in range(6)], device="cuda")).sum(dim=1)
    counts = torch.unique(code, return_counts=True)[1].double()
    assert counts.numel() == 720
    chi = float(((counts - n / 720) ** 2 / (n / 720)).sum().item())
    assert chi < 719 + 6 * (2 * 719) ** 0.5, chi
    # 3. the first card of a Klop deal is uniform over the legal set (12 cards, or 11 when the pagat is held)
    env.force_contract_synth(0)
    mask = env.mask[:n].clone()
    nleg = torch.zeros(n, dtype=torch.int64, device="cuda")
    for c in range(54):
        nleg += (mask >> c) & 1
    env.step_random(1)
    played = mask & ~env.hands[0, :n]                               # the card that left seat 0's hand
    below = torch.zeros(n, dtype=torch.int64, device="cuda")        # index of the played card inside the legal set
    seen = torch.zeros(n, dtype=torch.bool, device="cuda")
    for c in range(54):
        is_c = ((played >> c) & 1).bool()
        seen |= is_c
        below += (((mask >> c) & 1).bool() & ~seen).long()
    for k in (11, 12):
        sel = nleg == k
        cnt = torch.bincount(below[sel], minlength=k).double()
        m = float(sel.sum().item())
        chi = float(((cnt - m / k) ** 2 / (m / k)).sum().item())
        assert chi < (k - 1) + 6 * (2 * (k - 1)) ** 0.5, (k, chi)
    del hands, talon, order, mask
    env.close()
