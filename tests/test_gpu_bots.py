"""GPU: mixed tables -- Bot_igralec seats beside caller-driven (neural) seats, tarok_auction_bots / tarok_exchange_bots /
tarok_step_bots.

  * every seat a bot: deal + the three entries + score is bit for bit deal + auction_synth(18) + exchange_synth(0) +
    48 x step_random + score;
  * no bot: each entry is bit for bit its plain namesake on the same inputs;
  * mixed (a uniform seat mask per game, neural intents uniform in 0..19, neural exchanges and cards from a seeded host
    rule): every game replayed by the C oracle (syn_replay_bots), which draws the bots' decisions itself -- contract, king,
    exchange, the 48 plays and the scores agree game by game; the same with the lock-step specialisation or PDL off, with
    garbage card bytes for bot movers, and with games held back by TAROK_CARD_SKIP;
  * invalid inputs (mask bits 4-7, NULL / misaligned pointers) and Samoigra(boti=...).
Bar: bit-exact."""
import ctypes as C

import numpy as np
import pytest
import torch

import tarok_b200.env as E
from oracle import mixed

pytestmark = pytest.mark.gpu

SEED = 0xB0751
CARD_SKIP = 0xFE
DISCARDABLE = 0x7F7F7F7F | (0x3F << 33)
SIZES = [(1 << 20, 0), (1 << 20, 1001), (100003, 0), (100003, 77)]   # 100003: odd, not a multiple of the 512-game tile


def u64(t):
    return t.detach().cpu().numpy().view(np.uint64)


def state(env):
    """Every field a step can touch, by seat where the device keeps slots, plus the statistics vector."""
    n = env.n
    out = {f: getattr(env, f)[..., :n].clone() for f in ("meta", "piles", "talon", "mask", "hist", "discard")}
    out["hands"] = env.hands[:, :n].clone()
    out["scores"] = env.scores[:n].clone()
    out["stats"] = torch.from_numpy(env.stats())
    return out


def assert_same(a, b, what):
    for k in a:
        if not torch.equal(a[k].cpu(), b[k].cpu()):
            d = (a[k].cpu() != b[k].cpu())
            raise AssertionError("%s: %s differs (%d entries)" % (what, k, int(d.sum())))


def mix(gid, t, salt):
    """A seeded per-(game, play) hash on the device: int64 in [0, 2^31)."""
    h = (gid * 1000003 + t * 7919 + salt * 104729) & 0xFFFFFFF
    h = ((h ^ (h >> 11)) * 1274126177) & 0x7FFFFFFF
    return (h ^ (h >> 15)) & 0x7FFFFFFF


def nth_bit(m, r):
    """Card id of the r-th (0-based) set bit of every int64 bitboard m (54 when r >= popcount)."""
    bits = (m[:, None] >> torch.arange(54, device=m.device)[None, :]) & 1
    return (bits.cumsum(1) <= r[:, None]).sum(1)


def popcount(m):
    return ((m[:, None] >> torch.arange(54, device=m.device)[None, :]) & 1).sum(1)


def host_cards(env, gid, salt):
    """The neural players' rule: a seeded uniform pick among the mover's legal cards (env.mask), keyed by the play index."""
    mask = env.mask[:env.n]
    plays = E.meta_field(env.meta[:env.n], E.M_PLAYS, 6)
    cnt = popcount(mask)
    card = nth_bit(mask, mix(gid, plays, salt) % cnt.clamp(min=1))
    return torch.where(cnt > 0, card, torch.full_like(card, 0xFF)).to(torch.uint8)


def host_exchange(env, gid, salt):
    """The neural declarers' rule: a seeded group, then k seeded distinct discardable cards of hand + group."""
    n = env.n
    meta = env.meta[:n]
    contract = E.meta_field(meta, E.M_CONTRACT, 4)
    decl = E.meta_field(meta, E.M_DECL, 2)
    k = torch.tensor([0, 3, 2, 1, 3, 2, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0], device=meta.device)[contract]
    ngroups = torch.where(k > 0, 6 // k.clamp(min=1), torch.ones_like(k))
    group = mix(gid, 64, salt) % ngroups
    order = env.talon_order[:n]
    gb = torch.zeros_like(order)
    for j in range(3):
        cid = (order >> (6 * (group * k + j))) & 63
        gb |= torch.where(j < k, torch.ones_like(cid) << cid, torch.zeros_like(cid))
    hand = torch.gather(env.hands[:, :n], 0, decl[None, :])[0]
    avail = (hand | gb) & DISCARDABLE
    disc = torch.zeros_like(avail)
    for j in range(3):
        cnt = popcount(avail)
        c = nth_bit(avail, mix(gid, 65 + j, salt) % cnt.clamp(min=1))
        bit = torch.where((j < k) & (cnt > 0), torch.ones_like(c) << c.clamp(max=53), torch.zeros_like(c))
        disc |= bit
        avail &= ~bit
    return group.to(torch.uint8), disc


def bot_mover(env, bots):
    mover = (E.meta_field(env.meta[:env.n], E.M_LEADER, 2) + E.meta_field(env.meta[:env.n], E.M_POS, 2)) & 3
    return ((bots.to(torch.int64) >> mover) & 1).bool()


def play_mixed(n, first_gid, bots, intents, lockstep=True, pdl=True, garbage=0, skip=False):
    """deal -> auction_bots -> exchange_bots -> step_bots until every game is over -> score.  garbage = 0: bot movers get
    their own legal host pick; else a seeded byte in {0..53, 0xFF} (illegal ids included).  skip: a seeded third of the live
    games is held back by TAROK_CARD_SKIP at every launch.  Returns (env, perm, fed card per play [48, n])."""
    env = E.TarokEnv(n, seed=SEED, history=True)
    env.set_lockstep(lockstep)
    env.set_pdl(pdl)
    env.deal(first_gid)
    perm = env.export_perm()
    dev = env.torch_device
    gid = torch.arange(n, dtype=torch.int64, device=dev) + first_gid
    env.auction(intents, bots=bots)
    group, disc = host_exchange(env, gid, 3)
    env.exchange(group, disc, bots=bots)
    fed = torch.full((48, n), 0xFF, dtype=torch.uint8, device=dev)
    for launch in range(200):
        live = env.live()
        if not bool(live.any()):
            break
        cards = host_cards(env, gid, 5)
        if garbage:
            junk = mix(gid, launch, garbage) % 55
            junk = torch.where(junk == 54, torch.full_like(junk, 0xFF), junk).to(torch.uint8)
            cards = torch.where(bot_mover(env, bots), junk, cards)
        plays = E.meta_field(env.meta[:n], E.M_PLAYS, 6)
        if skip:
            cards = torch.where(mix(gid, launch, 9) % 3 == 0, torch.full_like(cards, CARD_SKIP), cards)
        moving = live & (cards != CARD_SKIP)
        fed[plays[moving], torch.nonzero(moving).flatten()] = cards[moving]
        env.step(cards, bots=bots)
    assert not bool(env.live().any())
    env.score()
    return env, perm, fed


def mixed_inputs(n, first_gid):
    rng = np.random.default_rng(first_gid + n)
    bots = torch.from_numpy(rng.integers(0, 16, n, dtype=np.uint8)).cuda()
    intents = torch.from_numpy(rng.integers(0, 20, (n, 4), dtype=np.uint8)).cuda()
    return bots, intents


# ---- every seat a bot / no bot -------------------------------------------------------------------------------------

@pytest.mark.parametrize("n,first_gid", SIZES)
def test_all_bots_is_the_mode_18_pipeline(n, first_gid):
    a = E.TarokEnv(n, seed=SEED, history=True)
    b = E.TarokEnv(n, seed=SEED, history=True)
    bots = torch.full((n,), 0x0F, dtype=torch.uint8, device=a.torch_device)
    junk = torch.randint(0, 256, (n, 4), dtype=torch.uint8, device=a.torch_device)      # bot intents are never read
    a.deal(first_gid); b.deal(first_gid)
    a.auction(junk, bots=bots); b.auction_synth(E.MODE_AUCTION_BOT)
    assert_same(state(a), state(b), "auction")
    a.exchange(torch.full((n,), 9, dtype=torch.uint8, device=a.torch_device), torch.full((n,), -1, dtype=torch.int64,
               device=a.torch_device), bots=bots)
    b.exchange_synth(False)
    assert_same(state(a), state(b), "exchange")
    cards = torch.full((n,), 0xFF, dtype=torch.uint8, device=a.torch_device)
    for t in range(48):
        a.step(cards, bots=bots)
        b.step_random()
    a.score(); b.score()
    sa, sb = state(a), state(b)
    assert_same(sa, sb, "after 48 steps and score")
    assert int(sa["stats"][E.S_FINISHED]) + int(sa["stats"][E.S_ERRORS]) == n


@pytest.mark.parametrize("n,first_gid", SIZES[1:3])
def test_no_bots_is_the_plain_entries(n, first_gid):
    a = E.TarokEnv(n, seed=SEED, history=True)
    b = E.TarokEnv(n, seed=SEED, history=True)
    dev = a.torch_device
    gid = torch.arange(n, dtype=torch.int64, device=dev) + first_gid
    zero = torch.zeros(n, dtype=torch.uint8, device=dev)
    _, intents = mixed_inputs(n, first_gid)
    intents[::97, 1] = 23                                                        # a few error games too
    a.deal(first_gid); b.deal(first_gid)
    a.auction(intents, bots=zero); b.auction(intents)
    assert_same(state(a), state(b), "auction")
    group, disc = host_exchange(a, gid, 3)
    group[::101] = 5                                                             # invalid groups / discards as well
    a.exchange(group, disc, bots=zero); b.exchange(group, disc)
    assert_same(state(a), state(b), "exchange")
    for t in range(48):
        cards = host_cards(a, gid, 5)
        cards[t::89] = 0xFF
        a.step(cards, bots=zero); b.step(cards)
        if t % 12 == 11:
            assert_same(state(a), state(b), "step %d" % t)
    a.score(); b.score()
    assert_same(state(a), state(b), "score")


# ---- mixed tables against the oracle ---------------------------------------------------------------------------------

def check_against_oracle(oracle, env, perm, fed, bots, intents, first_gid):
    n = env.n
    m = u64(env.meta[:n])
    f = lambda sh, b: ((m >> np.uint64(sh)) & np.uint64((1 << b) - 1)).astype(np.int64)
    hist = env.hist[:, :n].cpu().numpy().T                                      # [n, 48]
    cards = np.where(hist == 0xFF, 0xFF, hist & 63).astype(np.uint8)
    group = f(E.M_GROUP, 3)
    disc = u64(env.discard[:n])
    bots_np = bots.cpu().numpy()
    ref = mixed.replay_bots(SEED, first_gid, perm.cpu().numpy(), intents.cpu().numpy(), bots_np,
                             np.where(group == 7, 0xFF, group).astype(np.uint8), disc, cards)
    err = f(E.M_ERR, 1)
    np.testing.assert_array_equal(ref["mismatch"], -1, err_msg="bot plays differ from syn_play_draw")
    np.testing.assert_array_equal(ref["err"], err, err_msg="error games")
    ok = err == 0
    assert ok.mean() > 0.99
    np.testing.assert_array_equal(ref["contract"][ok], f(E.M_CONTRACT, 4)[ok], err_msg="contract")
    np.testing.assert_array_equal(ref["declarer"][ok], f(E.M_DECL, 2)[ok], err_msg="declarer")
    np.testing.assert_array_equal(ref["king"][ok], f(E.M_KING, 3)[ok], err_msg="king")
    exch = ok & (ref["group"] != 0xFF)
    np.testing.assert_array_equal(ref["group"][exch], group[exch], err_msg="group")
    np.testing.assert_array_equal(ref["discard"][exch], disc[exch], err_msg="discard")
    np.testing.assert_array_equal(ref["plays"][ok], cards[ok], err_msg="plays")
    np.testing.assert_array_equal(ref["scores"], env.scores[:n].cpu().numpy(), err_msg="scores")
    # the plays of the neural seats are the cards that were fed
    seat = np.where(hist == 0xFF, 0, hist >> 6)
    neural = (hist != 0xFF) & (((bots_np[:, None] >> seat) & 1) == 0)
    np.testing.assert_array_equal(cards[neural], fed.cpu().numpy().T[neural], err_msg="neural plays")
    # every contract kind occurs
    assert set(np.unique(ref["contract"][ok]).tolist()) == set(range(10))


@pytest.mark.parametrize("n,first_gid", SIZES)
def test_mixed_tables_against_oracle(oracle, n, first_gid):
    bots, intents = mixed_inputs(n, first_gid)
    env, perm, fed = play_mixed(n, first_gid, bots, intents)
    check_against_oracle(oracle, env, perm, fed, bots, intents, first_gid)
    want = state(env)
    # the same games with the lock-step specialisation off, with PDL off, with garbage card bytes for the bot movers
    # (0xFF and illegal ids among them), and with a third of the live games held back at every launch
    for kw in (dict(lockstep=False), dict(pdl=False, garbage=11), dict(garbage=12, skip=True)):
        if n != SIZES[0][0] and kw.get("skip"):
            continue
        env2, _, _ = play_mixed(n, first_gid, bots, intents, **kw)
        assert_same(state(env2), want, str(kw))
        env2.close()


# ---- invalid inputs -----------------------------------------------------------------------------------------------------

def test_skip_holds_bot_movers():
    n = 20000
    bots = torch.full((n,), 0x0F, dtype=torch.uint8, device="cuda")
    env = E.TarokEnv(n, seed=SEED, history=True)
    env.deal(3)
    env.auction(torch.zeros((n, 4), dtype=torch.uint8, device="cuda"), bots=bots)
    env.exchange(torch.zeros(n, dtype=torch.uint8, device="cuda"), torch.zeros(n, dtype=torch.int64, device="cuda"), bots=bots)
    before = state(env)
    env.step(torch.full((n,), CARD_SKIP, dtype=torch.uint8, device="cuda"), bots=bots)
    assert_same(state(env), before, "all skipped")
    half = torch.arange(n, device="cuda") % 2 == 0
    live = env.live()
    env.step(torch.where(half, CARD_SKIP, 0xFF).to(torch.uint8), bots=bots)
    plays = E.meta_field(env.meta[:n], E.M_PLAYS, 6)
    assert bool((plays[half] == 0).all())
    assert bool((plays[~half & live] == 1).all())


def test_mask_bits_above_seat_3_are_error_games():
    n = 30000
    dev = "cuda"
    env = E.TarokEnv(n, seed=SEED, history=True)
    gid = torch.arange(n, dtype=torch.int64, device=dev)
    bots, intents = mixed_inputs(n, 5)
    bad_a = torch.arange(n, device=dev) % 50 == 0
    env.deal(0)
    env.reset_stats()
    env.auction(intents, bots=torch.where(bad_a, bots | 0x10, bots))
    err = E.meta_field(env.meta[:n], E.M_ERR, 1).bool()
    assert bool(err[bad_a].all())
    assert int(env.stats()[E.S_ERR_EVENTS]) == int(err.sum())
    e0 = int(err.sum())
    waiting = E.meta_field(env.meta[:n], E.M_PHASE, 2) == E.PH_EXCHANGE
    bad_x = waiting & (torch.arange(n, device=dev) % 7 == 0)
    group, disc = host_exchange(env, gid, 3)
    env.exchange(group, disc, bots=torch.where(bad_x, bots | 0x80, bots))
    err = E.meta_field(env.meta[:n], E.M_ERR, 1).bool()
    assert bool(err[bad_x].all())
    e1 = int(err.sum())
    assert int(env.stats()[E.S_ERR_EVENTS]) == e1 and e1 >= e0 + int(bad_x.sum())
    live = env.live()
    bad_s = live & (torch.arange(n, device=dev) % 11 == 3)
    for t in range(2):                                  # counted once: the second launch finds the games over
        env.step(host_cards(env, gid, 5), bots=torch.where(bad_s, bots | 0x40, bots))
    err = E.meta_field(env.meta[:n], E.M_ERR, 1).bool()
    assert bool(err[bad_s].all())
    assert int(env.stats()[E.S_ERR_EVENTS]) == int(err.sum())


def test_null_and_misaligned_pointers_change_nothing():
    n = 5000
    env = E.TarokEnv(n, seed=SEED, history=True)
    lib, h, s = env._lib, env._h, env._stream()
    bots = torch.zeros(n + 8, dtype=torch.uint8, device="cuda")
    intents = torch.zeros((n, 4), dtype=torch.uint8, device="cuda")
    p = lambda t, off=0: C.c_void_p(t.data_ptr() + off)
    env.deal(0)
    before = state(env)
    assert lib.tarok_auction_bots(h, p(intents), None, s) < 0
    assert lib.tarok_auction_bots(h, p(intents, 1), p(bots), s) < 0
    assert_same(state(env), before, "auction_bots refused")
    env.auction(intents + 1, bots=bots[:n])
    before = state(env)
    group = torch.zeros(n, dtype=torch.uint8, device="cuda")
    disc = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    assert lib.tarok_exchange_bots(h, p(group), p(disc), None, s) < 0
    assert lib.tarok_exchange_bots(h, p(group), p(disc, 4), p(bots), s) < 0
    assert_same(state(env), before, "exchange_bots refused")
    env.exchange(group, disc[:n], bots=bots[:n] | 0x0F)
    before = state(env)
    cards = torch.zeros(n + 2, dtype=torch.uint8, device="cuda")
    assert lib.tarok_step_bots(h, p(cards), None, s) < 0
    assert lib.tarok_step_bots(h, p(cards), p(bots, 1), s) < 0
    assert lib.tarok_step_bots(h, p(cards, 1), p(bots), s) < 0
    assert_same(state(env), before, "step_bots refused")


# ---- Samoigra(boti=...) ---------------------------------------------------------------------------------------------------

def test_samoigra_all_bots_is_rollout_18():
    from tarok_b200.samoigra import Samoigra
    n = 65536
    s = Samoigra(n, seed=SEED, boti=(0, 1, 2, 3))
    assert s.mreze == [None] * 4
    st, _ = s.odigraj(first_game_id=1001)
    env = E.TarokEnv(n, seed=SEED)
    env.rollout(E.MODE_AUCTION_BOT, first_game_id=1001)
    np.testing.assert_array_equal(st, env.stats())
    assert list(s.vzorci(first_game_id=1001)) == []


def test_samoigra_without_bots_is_unchanged():
    from tarok_b200.mreze import ustvari_mreze
    from tarok_b200.samoigra import Samoigra
    n = 8192
    torch.manual_seed(3)
    mreze = [ustvari_mreze(torch.device("cuda")) for _ in range(4)]
    a = Samoigra(n, mreze=mreze, seed=SEED, random_card=[0.1, 0.2, 0.0, 0.3])
    b = Samoigra(n, mreze=mreze, seed=SEED, random_card=[0.1, 0.2, 0.0, 0.3], boti=())
    np.testing.assert_array_equal(a.odigraj(5)[0], b.odigraj(5)[0])


def test_samoigra_two_bots_against_oracle(oracle):
    from tarok_b200.samoigra import Samoigra
    n, fg = 65536, 12
    s = Samoigra(n, seed=SEED, boti=(2, 3), random_card=0.1)
    assert s.mreze[2] is None and s.mreze[3] is None
    st, _ = s.odigraj(first_game_id=fg)
    assert st[E.S_ERRORS] == 0 and st[E.S_ERR_EVENTS] == 0 and st[E.S_FINISHED] == n
    env = s.env
    m = u64(env.meta[:n])
    f = lambda sh, b: ((m >> np.uint64(sh)) & np.uint64((1 << b) - 1)).astype(np.uint8)
    # the deal as Igra.razdeli consumed it: each seat's dealt hand ascending, then the ordered talon
    h0 = u64(env.hands0[:, :n]).T
    bits = ((h0[:, :, None] >> np.arange(54, dtype=np.uint64)) & np.uint64(1)).astype(bool)
    hands = np.argsort(~bits, axis=2, kind="stable")[:, :, :12].reshape(n, 48)
    order = u64(env.talon_order[:n])
    talon = np.stack([(order >> np.uint64(6 * i)) & np.uint64(63) for i in range(6)], 1)
    perm = np.concatenate([hands, talon], 1).astype(np.uint8)
    hist = env.hist[:, :n].cpu().numpy().T
    cards = np.where(hist == 0xFF, 0xFF, hist & 63).astype(np.uint8)
    group = f(E.M_GROUP, 3)
    ref = oracle.replay(perm, f(E.M_CONTRACT, 4), f(E.M_DECL, 2), f(E.M_KING, 3), np.where(group == 7, 0xFF, group),
                        u64(env.discard[:n]), cards)
    np.testing.assert_array_equal(ref["err"], 0)
    np.testing.assert_array_equal(ref["scores"], env.scores[:n].cpu().numpy())
    # the bots' plays are syn_play_draw over the legal set the oracle computes at that play
    draw = oracle.lib().syn_play_draw
    draw.restype = C.c_uint32
    gid = np.arange(n, dtype=np.uint64) + np.uint64(fg)
    player = (ref["seat"].astype(np.int64) + gid[:, None].astype(np.int64)) % 4
    checked, sub = 0, 16384                       # the first 16384 games: one ctypes call per bot play
    for i, t in zip(*np.nonzero(((hist != 0xFF) & (player >= 2))[:sub])):
        mask = int(ref["mask"][i, t])
        r = draw(C.c_uint64(SEED), C.c_uint64(int(gid[i])), C.c_uint32(int(t)), C.c_uint32(bin(mask).count("1")))
        want = [c for c in range(54) if (mask >> c) & 1][r]
        assert cards[i, t] == want, (i, t)
        checked += 1
    assert checked > sub * 12                    # games that end early (Berac, Klop) play fewer than 48 cards
    # player sums by player: the bots are scored like everybody
    assert st[E.S_PLAYER:E.S_PLAYER + 4].sum() == st[E.S_SEAT:E.S_SEAT + 4].sum()
