"""GPU: BASELINE config 4 pipeline -- restated policy nets + device env / observations / action selection."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def test_neural_selfplay_rollout_is_legal_and_complete():
    import torch
    from tarok_b200.samoigra import Samoigra
    torch.manual_seed(0)
    n = 3000
    for eps in (0.0, 0.3):
        s = Samoigra(n, seed=77, random_card=eps)
        st, ms = s.odigraj(first_game_id=0, meri=True)
        assert st[18] + st[20] == n                       # every deal finished or was flagged ...
        assert st[20] <= 3 and st[21] == st[20]           # ... and only for Q19 hands (no illegal card ever selected)
        assert st[8:18].sum() == st[18]
        assert 10 * n < st[19] <= 48 * n                  # Berac games stop early
        assert set(ms) == {"env", "obs", "forward", "select", "bucket"}
        if eps > 0:
            assert (st[8:18] > 0).sum() >= 5              # exploring bids reach most contracts
        s.zapri()


def test_nets_follow_the_reference_call_contract():
    import torch
    from tarok_b200.mreze import ustvari_mreze
    nets = ustvari_mreze(torch.device("cuda"))
    B, T = 7, 16
    z = lambda *s: torch.zeros(s, device="cuda")
    for m in nets.values():
        m.eval()
    assert nets["Navadna_igra"]([z(B, T, 3, 54), z(B, 4), z(B, T, 54), z(B, 6, 55), z(B, 4), z(B, 54)]).shape == (B, 54)
    assert nets["Solo"]([z(B, T, 3, 54), z(B, T, 54), z(B, 6, 55), z(B, 4), z(B, 54)]).shape == (B, 54)
    assert nets["Klop"]([z(B, T, 3, 54), z(B, T, 54), z(B, 54)]).shape == (B, 54)
    assert nets["Berac"]([z(B, T, 3, 54), z(B, T, 54), z(B, 4)]).shape == (B, 54)
    assert nets["Vrednotenje_roke"](z(B, 54)).shape == (B, 18)
    assert nets["Zalaganje"]([z(B, 54), z(B, 54, 6), z(B, 15)]).shape == (B, 60)


def test_replay_samples_and_one_training_pass():
    import torch
    from tarok_b200.samoigra import Samoigra
    torch.manual_seed(1)
    n = 2048
    s = Samoigra(n, seed=5, random_card=0.2)
    st, _ = s.odigraj()
    total = 0
    for igralec, ime, T, stanje, dy in s.vzorci():
        assert 0 <= igralec < 4
        B = dy.shape[0]
        assert stanje[0].shape == (B, T, 3, 54) and dy.shape == (B, 54) and T % 8 == 0
        assert bool(((dy == -70) | (dy > -70)).all())
        total += B
    assert total == st[19]                                   # one sample per card play (Igralec.py:416)
    before = [p.detach().clone() for p in s.mreze[0]["Navadna_igra"].parameters()]
    loss = s.nauci()
    assert loss and all(np.isfinite(v) for v in loss.values())
    after = list(s.mreze[0]["Navadna_igra"].parameters())
    assert any(not torch.equal(a, b) for a, b in zip(before, after))
    s.zapri()


def _kopije(osnova, faktor):
    """A copy of the net set ``osnova`` whose six output layers are scaled by ``faktor`` (a power of two: exact in floating
    point): the argmax of every decision is unchanged bit for bit, and every recorded Q value tells which copy produced it."""
    import copy
    import torch
    d = copy.deepcopy(osnova)
    with torch.no_grad():
        for m in d.values():
            m.glava.izhod.weight *= faktor
            m.glava.izhod.bias *= faktor
    return d


def test_four_players_equal_single_player_runs_on_their_seats():
    """The reference seats four Nevronski_igralec with their own nets (main.py:48-66); player of seat s in game i = (s + i) % 4
    (Tarok.py:34).  Four copies of ONE net set, the copy of player p scaled by 2^p at the output, must play exactly the games
    four identical copies play, and the Q value recorded at every card play must be 2^p times the unscaled one for the player
    p that owned that seat: each decision was routed to its own player's network.  Against the single shared set (one
    player: larger forward batches, so the library LSTM / GEMM kernels may round differently) the games must agree too --
    exactly as a rule, and in any case for all but a handful of near-tie decisions."""
    import torch
    from tarok_b200.mreze import ustvari_mreze
    from tarok_b200.samoigra import Samoigra
    torch.manual_seed(3)
    n, seed, gid0 = 4096, 11, 5
    osnova = ustvari_mreze(torch.device("cuda"))
    a1 = Samoigra(n, mreze=osnova, seed=seed, random_card=0.1)                                    # one shared set
    a4 = Samoigra(n, mreze=[_kopije(osnova, 1.0) for _ in range(4)], seed=seed, random_card=[0.1] * 4)
    b = Samoigra(n, mreze=[_kopije(osnova, 2.0 ** p) for p in range(4)], seed=seed, random_card=[0.1] * 4)
    s1, _ = a1.odigraj(gid0)
    s4, _ = a4.odigraj(gid0)
    sb, _ = b.odigraj(gid0)
    h1, h4, hb = (x.env.hist[:, :n].cpu().numpy() for x in (a1, a4, b))
    # (1) routing: identical games, Q values scaled by the owner's factor
    assert (s4[:21] == sb[:21]).all()
    assert (h4 == hb).all()
    assert (a4.env.scores[:n].cpu().numpy() == b.env.scores[:n].cpu().numpy()).all()
    q4, qb = a4.env.qmax_hist[:, :n].cpu().numpy(), b.env.qmax_hist[:, :n].cpu().numpy()
    played = h4 != 0xFF
    seat = (h4 >> 6).astype(np.int64)
    player = (seat + (np.arange(n)[None, :] + gid0)) & 3
    assert played.sum() == s4[19]
    assert (qb[played] == q4[played] * (2.0 ** player[played]).astype(np.float32)).all()
    assert max(b.zadnji_koraki) > max(a1.zadnji_koraki)                           # more buckets: four players' queues
    # (2) the player-keyed bucketing does not change the games
    same = (h1 == h4).all(axis=0)
    assert same.mean() > 0.99, same.mean()
    if same.all():
        assert (s1[:21] == s4[:21]).all()
    a1.zapri(); a4.zapri(); b.zapri()


def test_device_buckets_match_the_host_partition():
    """tarok_obs_buckets == the (net, T) grouping obs_shape gives the host, keyed by the mover's player, in stable order."""
    import torch
    import tarok_b200.env as E
    n, gid0 = 20000, 123
    env = E.TarokEnv(n, seed=99, history=True)
    env.setup_synth(E.MODE_AUCTION_UNIFORM, gid0)
    for t in range(20):
        vrsta, vrstice = env.obs_shape()
        meta = env.meta[:n]
        mover = (E.meta_field(meta, E.M_LEADER, 2) + E.meta_field(meta, E.M_POS, 2)) & 3
        for players in (1, 4):
            sel, cnt = env.obs_buckets(players)
            cnt = cnt.copy()
            key = vrsta.to(torch.int64) * 7 + (vrstice.to(torch.int64) // 8 - 1)
            if players == 4:
                key = key + 28 * ((mover + torch.arange(n, device=meta.device) + gid0) & 3)
            live = vrsta != 255
            key = torch.where(live, key, torch.full_like(key, 127)).cpu().numpy()
            want = np.bincount(key[key != 127], minlength=128)[:128]
            assert (cnt[:128] == want).all() and cnt[127] == 0 and cnt[255] == want.sum()
            assert (cnt[128:256] == np.concatenate([[0], np.cumsum(want)[:-1]])).all()
            rows = want * (8 * (np.arange(128) % 7 + 1))
            assert (cnt[256:384] == np.concatenate([[0], np.cumsum(rows)[:-1]])).all()
            order = np.argsort(key, kind="stable")
            order = order[: int(want.sum())]
            assert (sel[: int(want.sum())].cpu().numpy() == order).all()
        del meta, mover, sel
        env.step_random()
    env.close()


def test_buckets_follow_the_first_game_id_of_every_deal():
    """One handle dealt again and again at first game ids of every residue mod 4 (and above 2^32): the bucket of each game
    is keyed by the player (mover + game id) % 4 of THAT deal.  The counting sort is replayed from a captured CUDA graph,
    which must not keep the rotation of the deal it was captured in."""
    import torch
    import tarok_b200.env as E
    n = 5000
    env = E.TarokEnv(n, seed=99, history=True)
    for gid0 in (0, 1, 2, 3, 6, 2 ** 32 + 1, 4):
        env.setup_synth(E.MODE_AUCTION_UNIFORM, gid0)
        for t in range(3):
            vrsta, vrstice = env.obs_shape()
            meta = env.meta[:n]
            mover = (E.meta_field(meta, E.M_LEADER, 2) + E.meta_field(meta, E.M_POS, 2)) & 3
            key = vrsta.to(torch.int64) * 7 + (vrstice.to(torch.int64) // 8 - 1)
            key = key + 28 * ((mover + torch.arange(n, device=meta.device) + gid0) & 3)
            key = torch.where(vrsta != 255, key, torch.full_like(key, 127)).cpu().numpy()
            sel, cnt = env.obs_buckets(4)
            want = np.bincount(key[key != 127], minlength=128)[:128]
            assert (cnt[:128] == want).all(), (gid0, t)
            assert (sel[: int(want.sum())].cpu().numpy() == np.argsort(key, kind="stable")[: int(want.sum())]).all()
            del meta, mover, sel
            env.step_random()
    env.close()


def test_all_bucket_launches_equal_the_per_bucket_kernels():
    """tarok_obs_expand_buckets / tarok_select_action_buckets (one launch for every bucket of a step) produce exactly what
    tarok_obs_expand / tarok_select_action produce bucket by bucket."""
    import torch
    import tarok_b200.env as E
    from tarok_b200.samoigra import _Arena
    n, gid0 = 6000, 77
    env = E.TarokEnv(n, seed=5, history=True)
    env.setup_synth(E.MODE_AUCTION_UNIFORM, gid0)
    ar = _Arena(n, env.torch_device)
    gen = torch.Generator(device=env.torch_device); gen.manual_seed(1)
    for t in range(14):
        sel, cnt = env.obs_buckets(4)
        cnt = cnt.copy()
        total = int(cnt[255])
        env.obs_expand_buckets(total, ar.opp, ar.hand, ar.talon, ar.talon_klop, ar.king, ar.decl, ar.disc)
        qs, cards_a, qmax_a = {}, torch.full((env.n_alloc,), 0xFF, dtype=torch.uint8, device="cuda"), torch.zeros(n, device="cuda")
        cards_b, qmax_b = cards_a.clone(), qmax_a.clone()
        for k in range(127):
            B, off, row = int(cnt[k]), int(cnt[128 + k]), int(cnt[256 + k])
            if not B:
                continue
            p, vr, T = k // 28, (k % 28) // 7, 8 * (k % 7 + 1)
            ref, ok = env.obs_expand(vr, T, sel[off:off + B])
            assert bool(ok.all())
            opp = ar.opp[row * 162:(row + B * T) * 162].view(B, T, 3, 54)
            hand = ar.hand[row * 54:(row + B * T) * 54].view(B, T, 54)
            assert torch.equal(opp, ref[0]) and torch.equal(hand, ref[2 if vr == 1 else 1])
            if vr == 0:
                assert torch.equal(ar.talon_klop[off * 54:(off + B) * 54].view(B, 54), ref[2])
            if vr in (1, 2):
                assert torch.equal(ar.talon[off * 330:(off + B) * 330].view(B, 6, 55), ref[3 if vr == 1 else 2])
                assert torch.equal(ar.disc[off * 54:(off + B) * 54].view(B, 54), ref[5 if vr == 1 else 4])
            if vr == 1:
                assert torch.equal(ar.king[off * 4:(off + B) * 4].view(B, 4), ref[1])
            if vr != 0:
                assert torch.equal(ar.decl[off * 4:(off + B) * 4].view(B, 4), ref[{1: 4, 2: 3, 3: 2}[vr]])
            qs[k] = torch.randint(0, 4, (B, 54), device="cuda", generator=gen).float()        # tie-prone outputs
            env.select_action(qs[k], sel[off:off + B], 0.2 * p, cards=cards_b, qmax=qmax_b)
        env.select_action_buckets(total, qs, [0.0, 0.2, 0.4, 0.6], cards_a, qmax_a)
        live = env.live()
        assert torch.equal(cards_a[:n][live], cards_b[:n][live]) and torch.equal(qmax_a[live], qmax_b[live])
        del live, sel
        env.step(cards_a)
    assert env.errors() <= 3
    env.close()
