"""CPU: the host helpers that tests/test_gpu_samoigra_reference.py judges whole Samoigra rollouts with.

  * ``nevronski.dense_batch`` (the vectorised input lists) equals ``nevronski.dense`` game by game at every play of oracle
    rollouts of each contract;
  * the stand-in networks of ``oracle/stub_nets.py`` give, in fp32, bf16 and fp16, exactly what they give in float64, and
    have the properties the rollout check relies on (every input, the row order, the player and ties all matter);
  * ``nevronski.exchange_observation`` has the layout ``k_obs_exchange`` documents (tarok_obs.cuh)."""
import numpy as np
import pytest
import torch

from oracle import nevronski as N
from oracle import stub_nets as S

SEED = 0x5EED0042AB
KINDS = {0: "Klop", 1: "Navadna_igra", 2: "Solo", 3: "Berac"}


@pytest.mark.parametrize("contract", range(10))
def test_dense_batch_is_dense_game_by_game(oracle, contract):
    n = 40
    r = oracle.rollout(SEED, contract & 1, n, contract)
    d = dict(perm=r["perm"], contract=r["contract"], declarer=r["declarer"], king=r["king"], group=r["group"],
             discard_mask=r["discard"], cards=r["cards"])
    L = oracle.lists(r["perm"], r["contract"], r["declarer"], r["king"], r["group"], r["discard"], r["cards"])
    seen = 0
    for t in range(48):
        o = N.observation(d, L, t)
        live = o["live"]
        for kind in range(4):
            for T in np.unique(o["T"][live & (o["kind"] == kind)]):
                games = np.nonzero(live & (o["kind"] == kind) & (o["T"] == T))[0]
                for with_mozne in (True, False):
                    got = N.dense_batch(o, games, with_mozne)
                    for i, g in enumerate(games):
                        want = N.dense(o, g, with_mozne)
                        assert len(got) == len(want)
                        for a, b in zip(got, want):
                            assert a.dtype == np.uint8 and np.array_equal(a[i], b), (t, kind, T, g)
                seen += len(games)
    assert seen > 10 * n                                  # Berac games may stop after one trick


def _inputs(rng, kind, B, T):
    """Random 0/1 input lists of one play net type (reference order)."""
    z = lambda *s: (rng.random(s) < 0.3).astype(np.uint8)
    return {0: [z(B, T, 3, 54), z(B, T, 54), z(B, 54)],
            1: [z(B, T, 3, 54), z(B, 4), z(B, T, 54), z(B, 6, 55), z(B, 4), z(B, 54)],
            2: [z(B, T, 3, 54), z(B, T, 54), z(B, 6, 55), z(B, 4), z(B, 54)],
            3: [z(B, T, 3, 54), z(B, T, 54), z(B, 4)]}[kind]


def _run(m, x, dtype):
    with torch.no_grad():
        if isinstance(x, list):
            y = m([torch.from_numpy(a).to(dtype) for a in x])
        else:
            y = m(torch.from_numpy(x).to(dtype))
    assert y.dtype == dtype
    return y.double().numpy()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_stub_nets_are_exact_in_every_dtype(dtype):
    """Every output of every player's six nets is the float64 one, on dense 0/1 inputs (30 % ones: far denser than any
    observation, so the sums are larger than in play)."""
    rng = np.random.default_rng(1)
    B = 96
    for p in range(4):
        nets = S.nets(p)
        for kind, name in KINDS.items():
            for T in (8, 24, 56):
                x = _inputs(rng, kind, B, T)
                want = S.host(nets[name], x)
                assert np.array_equal(_run(nets[name], x, dtype), want), (p, name, T)
                assert (want >= 0).all() and (want < S.MODULI[p]).all()
        hand = (rng.random((B, 54)) < 0.25).astype(np.uint8)
        assert np.array_equal(_run(nets["Vrednotenje_roke"], hand, dtype), S.host(nets["Vrednotenje_roke"], hand))
        ex = [(rng.random((B, 54)) < 0.25).astype(np.uint8), (rng.random((B, 54, 6)) < 0.1).astype(np.uint8),
              np.eye(15, dtype=np.uint8)[rng.integers(0, 15, B)]]
        assert np.array_equal(_run(nets["Zalaganje"], ex, dtype), S.host(nets["Zalaganje"], ex))


def _argmax_changes(a, b):
    return float((np.argmax(a, 1) != np.argmax(b, 1)).mean())


def test_stub_nets_see_every_input_the_row_order_and_the_player():
    rng = np.random.default_rng(2)
    B, T = 512, 24
    for kind, name in KINDS.items():
        x = _inputs(rng, kind, B, T)
        base = S.host(S.nets(1)[name], x)
        for j in range(len(x)):                            # each list entry on its own
            y = [a.copy() for a in x]
            y[j] = _inputs(rng, kind, B, T)[j]
            assert _argmax_changes(S.host(S.nets(1)[name], y), base) > 0.3, (name, j)
        for j in (0, 2 if kind == 1 else 1):               # opp / hand rows shifted by one (a wrong bucket offset)
            y = [a.copy() for a in x]
            y[j] = np.concatenate([y[j][:, 1:], np.zeros_like(y[j][:, :1])], axis=1)
            assert _argmax_changes(S.host(S.nets(1)[name], y), base) > 0.3, (name, j, "shift")
        # the same history with 8 padding rows more (the game put in the next T bucket)
        y = [np.concatenate([a, np.zeros_like(a[:, :8])], axis=1) if a.ndim >= 3 and a.shape[1] == T else a for a in x]
        assert _argmax_changes(S.host(S.nets(1)[name], y), base) > 0.3, (name, "T + 8")
        for p in (0, 2, 3):                                # another player decides differently
            assert _argmax_changes(S.host(S.nets(p)[name], x), base) > 0.3, (name, p)
    # king and decl (both [B,4] one-hots) swapped
    x = _inputs(rng, 1, B, T)
    x[1], x[4] = np.eye(4, dtype=np.uint8)[rng.integers(0, 4, B)], np.eye(4, dtype=np.uint8)[rng.integers(0, 4, B)]
    y = [x[0], x[4], x[2], x[3], x[1], x[5]]
    assert _argmax_changes(S.host(S.nets(0)["Navadna_igra"], y), S.host(S.nets(0)["Navadna_igra"], x)) > 0.3
    # bids and the exchange depend on the player
    hand = (rng.random((B, 54)) < 12 / 54).astype(np.uint8)
    ex = [hand, (rng.random((B, 54, 6)) < 0.02).astype(np.uint8), np.eye(15, dtype=np.uint8)[rng.integers(0, 15, B)]]
    for p in (0, 2, 3):
        assert _argmax_changes(S.host(S.nets(p)["Vrednotenje_roke"], hand), S.host(S.nets(1)["Vrednotenje_roke"], hand)) > 0.3
        a, b = S.host(S.nets(p)["Zalaganje"], ex), S.host(S.nets(1)["Zalaganje"], ex)
        assert _argmax_changes(a[:, 54:57], b[:, 54:57]) > 0.3 and _argmax_changes(a[:, :54], b[:, :54]) > 0.3


def test_stub_nets_tie_often_but_not_always():
    """Over 8 random legal cards, the top value is shared in a good fraction of decisions, but not in most."""
    rng = np.random.default_rng(3)
    B = 2000
    for p in range(4):
        q = S.host(S.nets(p)["Navadna_igra"], _inputs(rng, 1, B, 16))
        legal = np.argsort(rng.random((B, 54)), axis=1)[:, :8]
        v = np.take_along_axis(q, legal, axis=1)
        tied = ((v == v.max(1, keepdims=True)).sum(1) > 1).mean()
        assert 0.1 < tied < 0.8, (p, tied)


def test_exchange_observation_has_the_kernel_layout(oracle):
    """hand = the declarer's dealt cards; talon[card, group] = 1 for the six talon cards, group = position // k; game = the
    one-hot of igra_zalozi2index: Tri/Dve/Ena with king suit 0..3 -> 0..3 / 4..7 / 8..11, Solo_tri/dve/ena -> 12/13/14."""
    index = {(c, king): 4 * (c - 1) + king for c in (1, 2, 3) for king in range(4)}
    index.update({(4, None): 12, (5, None): 13, (6, None): 14})
    rng = np.random.default_rng(4)
    n = 240
    perm = oracle.deal(SEED, 7, n)
    contract = rng.integers(1, 7, n)
    declarer = rng.integers(0, 4, n)
    king = np.where(contract <= 3, rng.integers(0, 4, n), 0xFF)
    hand, talon, game = N.exchange_observation(perm, contract, declarer, king)
    assert hand.shape == (n, 54) and talon.shape == (n, 54, 6) and game.shape == (n, 15)
    for i in range(n):
        k = {1: 3, 2: 2, 3: 1, 4: 3, 5: 2, 6: 1}[int(contract[i])]
        want_h = np.zeros(54, np.uint8)
        want_h[perm[i, 12 * declarer[i]:12 * declarer[i] + 12]] = 1
        want_t = np.zeros((54, 6), np.uint8)
        for j in range(6):
            want_t[perm[i, 48 + j], j // k] = 1
        want_g = np.zeros(15, np.uint8)
        want_g[index[(int(contract[i]), int(king[i]) if contract[i] <= 3 else None)]] = 1
        assert np.array_equal(hand[i], want_h) and np.array_equal(talon[i], want_t) and np.array_equal(game[i], want_g), i
    assert talon.sum(axis=(1, 2)).tolist() == [6] * n and (talon.sum(1) > 0).sum(1).tolist() == (6 // np.array(
        [{1: 3, 2: 2, 3: 1, 4: 3, 5: 2, 6: 1}[int(c)] for c in contract])).tolist()
