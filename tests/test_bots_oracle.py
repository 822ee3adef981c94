"""Mixed tables in the C oracle (no GPU): ``syn_replay_bots`` with every seat a bot is the all-bot rollout of mode 18, with
no bot it is the fixed-intent auction, and ``Samoigra(boti=...)`` rejects bad arguments before it touches a device."""
import numpy as np
import pytest

from oracle import mixed

SEED = 0x5EED7A20C0001

# Nevronski_igralec.index2igra (0..17) + the two raw extras of the device's intents (18 Odprti_berac, 19 Klop) as Tip codes
TIP = np.array([-1] + [1] * 4 + [2] * 4 + [3] * 4 + [4, 5, 6, 7, 8, 9, 0], np.int8)


@pytest.mark.parametrize("first_gid", [0, 12345])
def test_all_bots_is_mode_18(oracle, first_gid):
    n = 12000
    ref = oracle.rollout(SEED, first_gid, n, oracle.MODE_AUCTION_BOT)
    intents = np.random.default_rng(first_gid).integers(0, 256, (n, 4), dtype=np.uint8)   # never read for a bot seat
    out = mixed.replay_bots(SEED, first_gid, ref["perm"], intents, np.full(n, 15, np.uint8), cards=ref["cards"])
    assert (out["mismatch"] == -1).all()
    np.testing.assert_array_equal(out["err"], ref["err"])
    np.testing.assert_array_equal(out["scores"], ref["scores"])
    np.testing.assert_array_equal(out["plays"], ref["cards"])
    ok = ref["err"] == 0
    for k in ("contract", "declarer", "king", "group", "discard"):
        np.testing.assert_array_equal(out[k][ok], ref[k][ok], err_msg=k)
    # the bot cards are drawn, not read: garbage in `cards` is reported, the game is the same
    bad = ref["cards"].copy()
    bad[:, 5] ^= 1
    out2 = mixed.replay_bots(SEED, first_gid, ref["perm"], intents, np.full(n, 15, np.uint8), cards=bad)
    np.testing.assert_array_equal(out2["plays"], ref["cards"])
    live5 = ref["cards"][:, 5] != 0xFF
    assert (out2["mismatch"][live5] == 5).all() and (out2["mismatch"][~live5] == -1).all()


def test_no_bots_is_the_fixed_intent_auction(oracle):
    n = 20000
    rng = np.random.default_rng(7)
    intents = rng.integers(0, 20, (n, 4), dtype=np.uint8)
    perm = oracle.deal(SEED, 0, n)
    out = mixed.replay_bots(SEED, 0, perm, intents, np.zeros(n, np.uint8))
    decl, contract, _ = oracle.auction_fixed(TIP[intents])
    np.testing.assert_array_equal(out["contract"], contract)
    np.testing.assert_array_equal(out["declarer"], decl)
    king_game = (contract >= 1) & (contract <= 3)
    suit = (intents[np.arange(n), decl].astype(np.int64) - 1) % 4
    np.testing.assert_array_equal(out["king"][king_game], suit[king_game])


def test_input_errors(oracle):
    n = 64
    perm = oracle.deal(SEED, 0, n)
    intents = np.full((n, 4), 1, np.uint8)
    bots = np.zeros(n, np.uint8)
    bots[:8] = 0x10 << np.arange(8) % 4                     # a bit above seat 3
    intents[8:16, 2] = 20                                   # past index 19 at a neural seat
    intents[16:24, 2] = 200
    bots[16:24] = 4                                         # ... at a bot seat: ignored
    out = mixed.replay_bots(SEED, 0, perm, intents, bots, cards=np.zeros((n, 48), np.uint8))
    assert out["err"][:16].all()
    assert (out["plays"][:16] == 0xFF).all()
    assert out["contract"][16:24].max() < 10


@pytest.mark.parametrize("kw", [dict(boti=(0,), igralci=1), dict(boti=(4,)), dict(boti=(-1,)), dict(boti=(1,), mreze={}),
                                dict(boti=("x",))])
def test_samoigra_rejects_bad_boti(kw):
    from tarok_b200.samoigra import Samoigra
    with pytest.raises(ValueError):
        Samoigra(16, **kw)
