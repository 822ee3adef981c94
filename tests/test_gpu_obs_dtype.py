"""GPU: bf16 / fp16 observations and selections (the *_ex entries of include/tarok_b200.h) against the fp32 entries.

Every observation value is 0 or 1, so a half observation must be the fp32 observation of the same call on the same state
converted, bit for bit; a selection on half network outputs must be the fp32 selection of the widened outputs (card, qmax,
qmax_hist, exploration, exchange group and discards).  The fp32 path itself is pinned to the float64 restatement of the
reference's player by test_gpu_neural_reference.py."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SEED = 0x5EED0042AB
HALF = ("bfloat16", "float16")
FILL = -1                                   # 0xFFFF as int16: the fill of half buffers before a call


def _dt(name):
    import torch
    return getattr(torch, name)


def _same(h, f):
    """half tensor == fp32 tensor converted, bit for bit."""
    import torch
    return torch.equal(h.view(torch.int16), f.to(h.dtype).view(torch.int16))


def _setup(n, mode, first_gid, exchange=True):
    from oracle import oracle as O
    from tarok_b200.env import TarokEnv
    r = O.rollout(SEED, first_gid, n, mode)
    env = TarokEnv(n, seed=SEED, history=True)
    env.set_deals(r["perm"], first_gid)
    env.force_contract(r["contract"], r["declarer"], r["king"])
    if exchange:
        env.exchange(r["group"], r["discard"])
    return env


def _ties(rng, n):
    import torch
    return torch.from_numpy(rng.integers(0, 3, (n, 54)).astype(np.float32))


# ---- 1. bucketed observations at every play ------------------------------------------------------------------------
ARENA = (("opp", 56 * 162), ("hand", 56 * 54), ("talon", 330), ("talon_klop", 54), ("king", 4), ("decl", 4), ("disc", 54))
WRITES = {"talon": (1, 2), "talon_klop": (0,), "king": (1,), "decl": (1, 2, 3), "disc": (1, 2)}    # net types per vector
GUARD = 64                                  # elements (128 bytes) after each half arena


@pytest.mark.parametrize("first_gid", [0, 1])
@pytest.mark.parametrize("mode", [16, 17, 18])
def test_bucketed_observations_every_play(mode, first_gid):
    """obs_expand_buckets into fp32, bf16 and fp16 arenas at every play of 65,536 games: every bucket's block matches, and
    what the call does not write (other net types' vectors, the tails, a guard after each arena) keeps its 0xFFFF fill."""
    import torch
    from tarok_b200.samoigra import _Arena
    n = 65536
    env = _setup(n, mode, first_gid)
    dev = env.torch_device
    f32 = _Arena(n, dev)
    half = {}
    for name in HALF:
        bufs = {a: torch.empty(n * per + GUARD, dtype=_dt(name), device=dev) for a, per in ARENA}
        half[name] = (bufs, {a: bufs[a][:n * per] for a, per in ARENA})
    rng = np.random.default_rng(mode * 2 + first_gid)
    steps = 0
    for t in range(48):
        if not bool(env.live().any()):
            break
        sel_dev, cnt = env.obs_buckets(4)
        total = int(cnt[255])
        env.obs_expand_buckets(total, f32.opp, f32.hand, f32.talon, f32.talon_klop, f32.king, f32.decl, f32.disc)
        keys = [k for k in range(127) if cnt[k]]
        rows = max(int(cnt[256 + k]) + int(cnt[k]) * 8 * (k % 7 + 1) for k in keys)
        net = (env._bk[3][:total].long() % 28) // 7                       # net type of every listed position
        for name in HALF:
            bufs, ar = half[name]
            for b in bufs.values():
                b.view(torch.int16).fill_(FILL)
            env.obs_expand_buckets(total, *[ar[a] for a, _ in ARENA])
            for a, per in ARENA:
                got = bufs[a].view(torch.int16)
                want = getattr(f32, a)
                if a in ("opp", "hand"):
                    m = rows * per // 56
                    assert _same(bufs[a][:m], want[:m]), (name, t, a)
                    assert bool((got[m:] == FILL).all()), (name, t, a, "tail")
                    continue
                written = torch.zeros(total, dtype=torch.bool, device=dev)
                for v in WRITES[a]:
                    written |= net == v
                g = got[:total * per].view(total, per)
                w = want[:total * per].view(total, per).to(_dt(name)).view(torch.int16)
                assert bool((g[written] == w[written]).all()), (name, t, a)
                assert bool((g[~written] == FILL).all()), (name, t, a, "other net types")
                assert bool((got[total * per:] == FILL).all()), (name, t, a, "tail")
        steps += 1
        order = sel_dev[:total].long()
        q = _ties(rng, n).to(dev)
        cards = torch.full((env.n_alloc,), 0xFF, dtype=torch.uint8, device=dev)
        env.select_action_buckets(total, {k: q[order[cnt[128 + k]:cnt[128 + k] + cnt[k]]].contiguous() for k in keys},
                                  [0.0] * 4, cards)
        env.step(cards)
    assert steps >= 40
    env.close()


# ---- 2. per-bucket observations --------------------------------------------------------------------------------------
def _obs_all_dtypes(env, kind, T, sel, play=None):
    import torch
    a32, ok32 = env.obs_expand(kind, T, sel, play=play)
    for name in HALF:
        ah, okh = env.obs_expand(kind, T, sel, play=play, dtype=_dt(name))
        assert torch.equal(okh, ok32), (name, kind, T, play)
        for x, y in zip(ah, a32):
            assert (x is None) == (y is None)
            if x is not None:
                assert x.dtype == _dt(name) and _same(x, y), (name, kind, T, play)
    return ok32


def test_per_bucket_observations_every_net_type():
    """obs_expand(net_type, T, sel) for the four net types at several plays of 65,536 mode-17 games: with sel=None (games
    of other buckets come out zero with ok = 0), with a shuffled selection that has repeats."""
    import torch
    n = 65536
    env = _setup(n, 17, 0)
    rng = np.random.default_rng(5)
    seen = set()
    for t in range(48):
        if not bool(env.live().any()):
            break
        if t in (0, 1, 9, 22, 35):
            kinds, rows = env.obs_shape()
            for kind in range(4):
                for T in torch.unique(rows[kinds == kind]).tolist():
                    ok = _obs_all_dtypes(env, kind, int(T), None)
                    assert bool(ok.any()) and not bool(ok.all())
                    sel = torch.from_numpy(rng.integers(0, n, 3000).astype(np.int32))
                    _obs_all_dtypes(env, kind, int(T), sel)
                    seen.add(kind)
        cards, _ = env.select_action(_ties(rng, n))
        env.step(cards)
    assert seen == {0, 1, 2, 3}
    env.close()


@pytest.mark.parametrize("contract", range(10))
def test_observations_as_of_every_play(contract):
    """obs_expand(..., play=t) for t = 0..47 on 8,192 finished games of each forced contract, at every T."""
    net = {0: 0, 1: 1, 2: 1, 3: 1, 4: 2, 5: 2, 6: 2, 7: 3, 8: 2, 9: 3}[contract]
    n = 8192
    env = _setup(n, contract, contract & 1)
    env.step_random(48)
    matched = 0
    for t in range(48):
        for T in range(8, 57, 8):
            matched += int(_obs_all_dtypes(env, net, T, None, play=t).sum())
    assert matched > 4 * n
    env.close()


# ---- 3. bidding and exchange observations ----------------------------------------------------------------------------
@pytest.mark.parametrize("mode", [16, 17])
def test_hand_and_exchange_observations(mode):
    import torch
    n = 65536
    env = _setup(n, mode, 0, exchange=False)
    h32 = env.obs_hands()
    (x32, ok32) = env.obs_exchange()
    for name in HALF:
        hh = env.obs_hands(_dt(name))
        assert hh.dtype == _dt(name) and _same(hh, h32), name
        xh, okh = env.obs_exchange(dtype=_dt(name))
        assert torch.equal(okh, ok32)
        for a, b in zip(xh, x32):
            assert _same(a, b), name
        sel = torch.from_numpy(np.random.default_rng(mode).integers(0, n, 5000).astype(np.int32))
        xs, _ = env.obs_exchange(sel, dtype=_dt(name))
        for a, b in zip(xs, x32):
            assert _same(a, b[sel.long().to(b.device)]), name
    assert bool(ok32.any())
    env.close()


# ---- 4. card and exchange choice on half outputs ---------------------------------------------------------------------
REGIMES = ("ties", "rounded", "zeros", "wide", "neg_inf", "nan_one", "all_nan")


def _q_half(rng, regime, n, legal, name):
    """[n,54] outputs of one regime in dtype `name`; `legal` (uint64 [n]) places the NaN of "nan_one" on a legal card."""
    import torch
    dt = _dt(name)
    if regime == "ties":
        return torch.from_numpy(rng.integers(0, 3, (n, 54)).astype(np.float32)).to(dt)
    if regime == "rounded":                                      # distinct fp32 values that round to equal half values
        return torch.from_numpy((rng.random((n, 54)) * 4).astype(np.float32)).to(dt)
    if regime == "zeros":
        return torch.from_numpy(np.where(rng.random((n, 54)) < 0.5, np.float32(0.0), np.float32(-0.0))).to(dt)
    if regime in ("wide", "nan_one"):
        bits = rng.integers(0, 1 << 16, (n, 54)).astype(np.uint16)           # every finite value, subnormals included
        q = torch.from_numpy(bits.view(np.int16)).view(dt).clone()
        fin = torch.finfo(dt)
        q[~torch.isfinite(q)] = 0
        pick = torch.from_numpy(rng.random((n, 54)))
        q[pick < 0.05] = fin.max
        q[pick > 0.95] = -fin.max
        small = (pick > 0.4) & (pick < 0.45)
        q[small] = torch.from_numpy(rng.integers(-3, 3, int(small.sum()))).to(dt)
        sub = (pick > 0.45) & (pick < 0.5)
        q[sub] = (torch.from_numpy(rng.integers(1, 4, int(sub.sum()))).to(dt) * fin.smallest_normal / 4).to(dt)
        if regime == "nan_one":
            b = ((np.asarray(legal, np.uint64)[:, None] >> np.arange(54, dtype=np.uint64)) & np.uint64(1)).astype(bool)
            cnt = b.sum(1)
            r = (rng.random(n) * np.maximum(cnt, 1)).astype(np.int64)
            at = np.argmax(b & (np.cumsum(b, 1) == r[:, None] + 1), axis=1)
            rows = np.nonzero(cnt)[0]
            q[torch.from_numpy(rows), torch.from_numpy(at[rows])] = float("nan")
        return q
    if regime == "neg_inf":
        q = torch.full((n, 54), float("-inf"), dtype=dt)
        q[torch.from_numpy(rng.random(n) < 0.3)] = -torch.finfo(dt).max
        return q
    if regime == "all_nan":
        return torch.full((n, 54), float("nan"), dtype=dt)
    raise ValueError(regime)


def _u32(x):
    import torch
    return x.view(torch.int32)


@pytest.mark.parametrize("name", HALF)
@pytest.mark.parametrize("variant", ["plain", "tab"])
def test_card_choice_on_half_outputs(variant, name):
    """Two identical environments, one fed the half outputs and one their fp32 widening, at eps 0 / 0.3 / 1: card, qmax
    and qmax_hist equal at every step of every regime (so is every exploration decision)."""
    import torch
    n, mode = 4096, 17
    rng = np.random.default_rng(["plain", "tab"].index(variant) * 2 + HALF.index(name))
    subnormal_seen = 0
    for regime in REGIMES:
        for eps, first_gid in ((0.0, 0), (0.3, 1), (1.0, 2)):
            envs = [_setup(n, mode, first_gid) for _ in range(2)]
            dev = envs[0].torch_device
            for t in range(48):
                live = envs[0].live()
                if not bool(live.any()):
                    break
                legal = envs[0].mask[:n].cpu().numpy().view(np.uint64)
                qh = _q_half(rng, regime, n, legal, name).to(dev)
                subnormal_seen += int(((qh != 0) & (qh.abs() < torch.finfo(qh.dtype).smallest_normal)).sum())
                out = []
                for env, q in zip(envs, (qh, qh.float())):
                    cards = torch.full((env.n_alloc,), 0xFF, dtype=torch.uint8, device=dev)
                    qm = torch.zeros(n, dtype=torch.float32, device=dev)
                    if variant == "plain":
                        sel = torch.nonzero(live).flatten().to(torch.int32)
                        env.select_action(q[sel.long()], sel, eps, cards, qm)
                    else:
                        sel_dev, cnt = env.obs_buckets(4)
                        total = int(cnt[255])
                        order = sel_dev[:total].long()
                        env.select_action_buckets(total, {k: q[order[cnt[128 + k]:cnt[128 + k] + cnt[k]]].contiguous()
                                                          for k in range(127) if cnt[k]}, [eps] * 4, cards, qm)
                    out.append((cards.clone(), qm.clone()))
                    env.step(cards)
                assert torch.equal(out[0][0], out[1][0]), (regime, eps, t, "card")
                assert torch.equal(_u32(out[0][1]), _u32(out[1][1])), (regime, eps, t, "qmax")
            played = envs[0].hist[:, :n] != 0xFF
            assert torch.equal(envs[0].hist[:, :n], envs[1].hist[:, :n]) and envs[0].errors() == envs[1].errors()
            assert torch.equal(_u32(envs[0].qmax_hist[:, :n])[played], _u32(envs[1].qmax_hist[:, :n])[played]), (regime, eps)
            for env in envs:
                env.close()
    assert subnormal_seen > 0


@pytest.mark.parametrize("name", HALF)
def test_exchange_choice_on_half_outputs(name):
    import torch
    n = 16384
    rng = np.random.default_rng(40 + HALF.index(name))
    for regime in REGIMES:
        for eps, first_gid in ((0.0, 0), (0.3, 1), (1.0, 2)):
            env = _setup(n, 17, first_gid, exchange=False)
            _, ok = env.obs_exchange()
            ex = torch.nonzero(ok).flatten().to(torch.int32)
            m = int(ex.numel())
            p = torch.cat([_q_half(rng, regime, m, np.zeros(m, np.uint64), name),
                           _q_half(rng, regime, m, np.zeros(m, np.uint64), name)[:, :6]], dim=1)
            if regime == "nan_one":
                p[torch.arange(m), torch.from_numpy(rng.integers(0, 54, m))] = float("nan")
                p[torch.arange(m), torch.from_numpy(54 + rng.integers(0, 2, m))] = float("nan")
            gh, dh = env.select_exchange(p, ex, eps)
            gf, df = env.select_exchange(p.float(), ex, eps)
            assert torch.equal(gh, gf) and torch.equal(dh, df), (regime, eps)
            assert bool((gh[ex.long()] != 0xFF).all())
            env.close()


# ---- 5. invalid inputs -----------------------------------------------------------------------------------------------
def test_invalid_inputs_are_errors_and_write_nothing():
    import torch
    from tarok_b200 import _lib
    n = 4096
    env = _setup(n, 17, 0)
    dev = env.torch_device
    sel_dev, cnt = env.obs_buckets(4)
    total = int(cnt[255])
    lib, p = env._lib, (lambda t: C.c_void_p(t.data_ptr()))

    def fresh(dt):
        return {a: torch.full((n * per + 16,), FILL, dtype=torch.int16, device=dev).view(dt) for a, per in ARENA}

    def untouched(bufs):
        torch.cuda.synchronize()
        return all(bool((b.view(torch.int16) == FILL).all()) for b in bufs.values())

    # an unknown dtype, at every new entry
    bufs = fresh(torch.bfloat16)
    sel, _, _, selkey = env._bk[:4]
    for dtype in (3, -1):
        assert lib.tarok_obs_expand_buckets_ex(env._h, dtype, p(sel), p(selkey), p(cnt_dev(env)), total,
                                               *[p(bufs[a]) for a, _ in ARENA], env._stream()) != 0
        assert lib.tarok_obs_expand_at_ex(env._h, dtype, -1, 1, 8, None, n, p(bufs["opp"]), p(bufs["hand"]), p(bufs["talon"]),
                                          p(bufs["king"]), p(bufs["decl"]), p(bufs["disc"]), p(bufs["talon_klop"]), None,
                                          env._stream()) != 0
        assert lib.tarok_obs_hands_ex(env._h, dtype, p(bufs["opp"]), env._stream()) != 0
        assert lib.tarok_obs_exchange_ex(env._h, dtype, None, n, p(bufs["hand"]), p(bufs["opp"]), p(bufs["disc"]), None,
                                         env._stream()) != 0
        assert b"dtype" in lib.tarok_last_error(env._h)
    assert untouched(bufs)
    cards = torch.full((env.n_alloc,), 0xFE, dtype=torch.uint8, device=dev)
    grp = torch.full((n,), 0xFE, dtype=torch.uint8, device=dev)
    disc = torch.full((n,), 7, dtype=torch.int64, device=dev)
    q = torch.zeros((n, 60), dtype=torch.bfloat16, device=dev)
    tab = (C.c_void_p * 128)()
    eps = (C.c_float * 4)(0.0, 0.0, 0.0, 0.0)
    for dtype in (3, -1):
        assert lib.tarok_select_action_ex(env._h, dtype, p(q), None, n, 0.0, p(cards), None, env._stream()) != 0
        assert lib.tarok_select_action_buckets_tab_ex(env._h, dtype, tab, p(sel), p(selkey), p(cnt_dev(env)), total, eps,
                                                      p(cards), None, env._stream()) != 0
        assert lib.tarok_select_exchange_ex(env._h, dtype, p(q), None, n, 0.0, p(grp), p(disc), env._stream()) != 0
    torch.cuda.synchronize()
    assert bool((cards == 0xFE).all()) and bool((grp == 0xFE).all()) and bool((disc == 7).all())

    # half arenas misaligned by 2 bytes
    for name in HALF:
        for a in ("opp", "hand", "talon", "talon_klop", "king", "decl", "disc"):
            bufs = fresh(_dt(name))
            args = {b: bufs[b][:n * per] for b, per in ARENA}
            args[a] = bufs[a][1:1 + n * dict(ARENA)[a]]
            with pytest.raises(_lib.TarokLibraryError, match="aligned"):
                env.obs_expand_buckets(total, *[args[b] for b, _ in ARENA])
            assert untouched(bufs), (name, a)
        bufs = fresh(_dt(name))
        with pytest.raises(_lib.TarokLibraryError, match="aligned"):
            lib_rc = lib.tarok_obs_expand_at_ex(env._h, HALF.index(name) + 1, -1, 1, 8, None, n, p(bufs["opp"][1:]),
                                                p(bufs["hand"]), None, None, None, None, None, None, env._stream())
            env._check(lib_rc)
        assert untouched(bufs)

    # mixed dtypes from Python
    ar = {a: torch.full((n * per,), FILL, dtype=torch.int16, device=dev).view(torch.float16) for a, per in ARENA}
    ar["king"] = torch.full((n * 4,), FILL, dtype=torch.int16, device=dev).view(torch.bfloat16)
    with pytest.raises(ValueError, match="mix"):
        env.obs_expand_buckets(total, *[ar[a] for a, _ in ARENA])
    assert untouched(ar)
    f64 = {a: torch.zeros(n * per, dtype=torch.float64, device=dev) for a, per in ARENA}
    with pytest.raises(ValueError):
        env.obs_expand_buckets(total, *[f64[a] for a, _ in ARENA])
    order = sel_dev[:total].long()
    qd = torch.zeros((n, 54), dtype=torch.float32, device=dev)
    keys = [k for k in range(127) if cnt[k]]
    assert len(keys) > 1
    mixed = {k: qd[order[cnt[128 + k]:cnt[128 + k] + cnt[k]]].to(torch.bfloat16 if i % 2 else torch.float16).contiguous()
             for i, k in enumerate(keys)}
    with pytest.raises(ValueError, match="mix"):
        env.select_action_buckets(total, mixed, [0.0] * 4, cards)
    torch.cuda.synchronize()
    assert bool((cards == 0xFE).all())
    with pytest.raises(ValueError):
        env.obs_hands(torch.float64)
    env.close()


def cnt_dev(env):
    return env._bk[1]


# ---- 6. end to end through Samoigra ----------------------------------------------------------------------------------
class _Stub:
    """Parameter-free nets whose outputs are small integers (exact in bf16 and fp16) computed from their inputs in the
    input dtype: counts over the opponents' rows plus three times the last hand row, plus the per-game vectors."""

    @staticmethod
    def nets(salt):
        import torch
        from torch import nn

        class Igra(nn.Module):
            def forward(self, x):
                opp, hand, rest = x[0], x[2] if len(x) == 6 else x[1], x[1:]
                y = opp.sum(dim=(1, 2)) + 3 * hand[:, -1] + salt * hand.sum(1)
                for v in rest:
                    if v.dim() == 2 and v.shape[1] == 54:
                        y = y + 2 * v
                    elif v.dim() == 2 and v.shape[1] == 4:                 # which of the four is set
                        w = torch.arange(1, 5, device=v.device, dtype=v.dtype)
                        y = y + ((v * w).sum(1, keepdim=True) + torch.arange(54, device=v.device, dtype=v.dtype)) % 7
                return y

        class Roka(nn.Module):
            def forward(self, x):
                return x[:, :18] * (1 + salt) + x[:, 18:36] * 2 + x[:, 36:54]

        class Zalaganje(nn.Module):
            def forward(self, x):
                hand, talon, game = x
                return torch.cat([hand + talon.sum(2) * 3 + salt, talon.sum(1) + game[:, :6] * 2], dim=1)

        return {"Navadna_igra": Igra(), "Klop": Igra(), "Solo": Igra(), "Berac": Igra(), "Vrednotenje_roke": Roka(),
                "Zalaganje": Zalaganje()}


def _play(dtype, mreze, n, seed):
    import torch
    from tarok_b200.samoigra import Samoigra
    s = Samoigra(n, mreze=mreze, seed=seed, random_card=[0.05] * 4, dtype=dtype)
    st, _ = s.odigraj(first_game_id=3)
    env = s.env
    out = dict(stats=st, scores=env.scores[:n].cpu().clone(), hist=env.hist[:, :n].cpu().clone(),
               hands0=env.hands0.cpu().clone())
    s.zapri()
    torch.cuda.synchronize()
    return out


def test_samoigra_half_plays_the_fp32_games():
    """Stub nets whose decisions depend on the arenas and the bucket offsets: Samoigra in bf16 and fp16 plays exactly the
    games of Samoigra in fp32 (same seed, eps 0.05): stats, scores, history and hands as dealt."""
    import torch
    n = 16384
    mreze = [_Stub.nets(p) for p in range(4)]
    ref = _play(torch.float32, mreze, n, 91)
    assert ref["stats"][18] == n
    for name in HALF:
        got = _play(_dt(name), mreze, n, 91)
        assert np.array_equal(got["stats"], ref["stats"]), name
        for k in ("scores", "hist", "hands0"):
            assert torch.equal(got[k], ref[k]), (name, k)


@pytest.mark.parametrize("name", ("float32",) + HALF)
def test_samoigra_real_nets_in_every_dtype(name):
    """Random-init nets, each dtype: every game finishes; the only error games are hands that cannot discard (Q19), never
    an illegal card.  The master nets stay fp32."""
    import torch
    from tarok_b200.samoigra import Samoigra
    n = 4096
    s = Samoigra(n, seed=12, dtype=_dt(name))
    for _ in range(2):
        st, ms = s.odigraj(meri=True)
        assert st[18] + st[20] == n and st[20] == st[21] and st[20] <= 3, (name, st[18], st[20], st[21])
        assert set(ms) >= {"env", "bucket", "obs", "select", "forward"}
    assert all(p.dtype == torch.float32 for d in s.mreze for m in d.values() for p in m.parameters())
    s.zapri()
