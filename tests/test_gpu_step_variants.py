"""GPU: the two persistent play_step kernels where each CTA loops over several 512-game tiles, against the C oracle and
against the plain kernel.

TAROK_OPT_STEP_IMPL = 2 launches k_step_tma on min(tiles, 4 x SMs) CTAs; 3 launches k_step_pp, for the interior launches of
a lock-step random chain with the draw cache on all three positions, on min(tiles, 5 x SMs) CTAs at trick positions 0-2 and
min(tiles, 4 x SMs) at position 3 (tarok_abi.cu, launch_step).  Each CTA prefetches tile + gridDim.x into the other of two
shared-memory stages and waits on that stage's mbarrier with parity (it >> 1) & 1, so a second iteration uses stage 1 and a
third reuses stage 0 with the flipped parity.  Below one wave (test_every_play_step_variant_matches_oracle) none of that
runs.  The sizes here come from the SM count of the device, so every case reaches the loop depth it names:

    A  4S + 1 tiles      k_step_tma and k_step_pp at position 3 take a second tile (stage 1)
    B  10S + 1 tiles     every persistent grid makes 3 iterations (stage 0 again, parity 1)
    C  1,048,576 deals   bench.py config 2 and tools/step_ab.py's 1 M size
    D  2^23 + 4,097      the 8 M A/B size: 22-28 iterations on a 148-SM B200; the draw cache is off there by default

A and B are ragged (the last tile holds padding games).  A profiler trace of each variant's first run proves which kernels
ran, on which grid, and so how many tiles a CTA took.  Every game is compared with the oracle (scores, cards, plays, error
bits, statistics); the chains, the desynchronised batch and the external cards are also compared, launch by launch, with a
handle that runs the plain kernel (TAROK_OPT_STEP_IMPL = 1) on the same inputs.  Bar: bit-exact."""
import json
import re

import pytest
import torch

pytestmark = pytest.mark.gpu

TILE = 512
SEED = 0x5EED57E9
GIDS = (2 ** 33 + 6, 12345)                   # even: k_step_pp reads the draw cache; odd: it computes every draw
MODES = (16, 17, 0)                           # lock-step throughout / Berac early stops and desynchronised tiles / Klop talon
CHAIN = (1, 2, 5, 3, 13, 1, 23)               # random chains whose ends switch kernels in the middle of a trick
DESYNC_CHAIN = (21, 27)                       # the 48 launches after the exchange of the desynchronised batch
STATE = ("meta", "hand_slots", "mask", "talon", "talon_order", "hist")
CARD_SKIP = 0xFE                              # TAROK_CARD_SKIP
PER_SM = {"tma": 4, "pp012": 5, "pp3": 4}     # resident CTAs per SM of the persistent grids (launch_step, TK_PP_BLOCKS_*)
# iterations the busiest CTA of each persistent grid makes, where they do not depend on the SM count (A, B); C and D only
# claim at least three, i.e. a stage reused under parity 1
ITERS = {"A": {"tma": 2, "pp012": 1, "pp3": 2}, "B": {"tma": 3, "pp012": 3, "pp3": 3}}
CASES = ("A", "B", "C", "D")


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def case_size(case, S):
    if case == "A":
        return (4 * S + 1) * TILE - 5
    if case == "B":
        return (10 * S + 1) * TILE - 37
    if case == "C":
        return 1 << 20
    return (1 << 23) + 4097


_ORACLE = {}


def reference(oracle, n, mode, gid):
    """The oracle's games (seed SEED, game ids gid ..), on the device.  Computed once per (size, mode, game id); only the
    current size is kept."""
    key = (n, mode, gid)
    if key not in _ORACLE:
        for k in [k for k in _ORACLE if k[0] != n]:
            del _ORACLE[k]
        r = oracle.rollout(SEED, gid, n, mode)
        _ORACLE[key] = dict(stats=oracle.device_stats(r), scores=torch.from_numpy(r["scores"]).cuda(),
                            cards=torch.from_numpy(r["cards"]).cuda(), plays=torch.from_numpy(r["plays"]).cuda().long(),
                            err=torch.from_numpy(r["err"]).cuda().long())
    return _ORACLE[key]


def assert_none(bad, what):
    if bool(bad.any()):
        idx = torch.nonzero(bad).flatten()
        raise AssertionError("%s: %d games differ, first %s" % (what, idx.numel(), idx[:8].tolist()))


def check_oracle(env, ref, what):
    """Statistics, and every game's scores, plays, error bit and cards, equal to the oracle's."""
    import tarok_b200.env as E
    n = env.n
    st = env.stats()[:21]
    assert (st == ref["stats"]).all(), "%s: stats %s != oracle %s" % (what, st.tolist(), ref["stats"].tolist())
    assert_none((env.scores[:n] != ref["scores"]).any(1), what + ": scores")
    meta = env.meta[:n]
    assert_none(((meta >> E.M_PLAYS) & 63) != ref["plays"], what + ": plays")
    assert_none(((meta >> E.M_ERR) & 1) != ref["err"], what + ": error bits")
    hist, cards = env.hist[:, :n].T, ref["cards"]
    assert_none(torch.where(cards != 0xFF, (hist & 63) != cards, hist != 0xFF).any(1), what + ": cards")


def check_same(a, b, what, fields=STATE):
    """The whole state of two handles, padding games included, is the same."""
    for f in fields:
        x, y = getattr(a, f), getattr(b, f)
        if not torch.equal(x, y):
            col = (x != y).reshape(-1, x.shape[-1]).any(0) if f != "scores" else (x != y).any(1)
            assert_none(col, "%s: %s differs from the plain kernel's" % (what, f))


def force_graph(env):
    """TAROK_OPT_GRAPH = 2: the stepwise rollout replays its CUDA graph at every batch size."""
    env._check(env._lib.tarok_set_option(env._h, 8, 2))


# ---- which kernels ran: torch.profiler trace --------------------------------------------------------------------------

STEP_KERNEL = re.compile(r"\bk_step(_tma|_pp)?<([^>]*)>")


def step_launches(fn, path):
    """Runs fn() under the profiler; returns (kernel, template arguments, grid.x) of every play_step launch in the trace."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    prof.export_chrome_trace(str(path))
    with open(path) as f:
        events = json.load(f)["traceEvents"]
    out = []
    for e in events:
        m = STEP_KERNEL.search(e.get("name", "")) if e.get("cat") == "kernel" else None
        if m:
            out.append(({"_tma": "tma", "_pp": "pp"}.get(m.group(1), "plain"), m.group(2).replace(" ", ""),
                        int(e["args"]["grid"][0])))
    return out


def pp_launches(chains, plays=0):
    """How many launches of these random chains take k_step_pp (launch_step): the interior launches of a chain while the
    host knows the lock-step play count, which it forgets after 48 launches."""
    k = 0
    for c in chains:
        for t in range(c):
            k += t + 1 < c and plays >= 0
            plays = plays + 1 if 0 <= plays < 47 else -1
    return k


SEEN = {}                                     # (case, kernel) -> (grid, tiles): what the traces showed


def check_launches(launches, case, impl, total, pp, graph, plain=0, random=True, what=""):
    """`total` play_step launches of the handle under test -- of which `pp` are k_step_pp (impl 3, kernel variant `graph`),
    or all are k_step_tma (impl 2) -- each on its persistent grid, with the iteration count the case claims, and `plain`
    launches of the plain kernel by the reference handle."""
    S = sms()
    tiles = (case_size(case, S) + TILE - 1) // TILE
    kinds = [k for k, _, _ in launches]
    want = {"tma": total if impl == 2 else 0, "pp": pp if impl == 3 else 0}
    want["plain"] = total + plain - want["tma"] - want["pp"]
    got = {k: kinds.count(k) for k in want}
    assert got == want, "%s: play_step launches %s, want %s" % (what, got, want)
    for kind, args, grid in launches:
        if kind == "plain":
            assert grid == tiles, what
            continue
        if kind == "tma":
            key = "tma"
            assert args == ("true" if random else "false"), (what, args)
        else:
            pos, g = args.split(",")
            key = "pp3" if pos == "3" else "pp012"
            assert g == ("true" if graph else "false"), (what, args)
        assert grid == min(tiles, PER_SM[key] * S), "%s: %s grid %d, tiles %d, %d SMs" % (what, key, grid, tiles, S)
        iters = -(-tiles // grid)
        if case in ITERS:
            assert iters == ITERS[case][key], (what, key, grid, tiles)
        else:
            assert iters >= 3, (what, key, grid, tiles)
        if case != "A":
            assert tiles > 2 * grid, (what, key, grid, tiles)
        SEEN[(case, key)] = (grid, tiles, iters)


# ---- the entries ------------------------------------------------------------------------------------------------------

def chains(t, r, chunks, what):
    for i, c in enumerate(chunks):
        t.step_random(c)
        r.step_random(c)
        check_same(t, r, "%s, chunk %d (%d steps)" % (what, i, c))


def score_both(t, r, ref, what):
    t.score()
    r.score()
    check_same(t, r, what, ("piles", "scores"))
    check_oracle(t, ref, what)


def run_chain(t, r, mode, gid, ref, what):
    t.reset_stats(); r.reset_stats()
    t.setup_synth(mode, gid); r.setup_synth(mode, gid)
    check_same(t, r, what + ", setup")
    chains(t, r, CHAIN, what)
    score_both(t, r, ref, what)


def run_desync(t, r, gid, ref, what):
    """Mode 17 as in test_desynchronised_batch_takes_the_general_path: the contracts without a talon exchange play two
    cards before the others have exchanged, so the lock-step hint is wrong for part of most warps."""
    for e in (t, r):
        e.reset_stats()
        e.deal(gid)
        e.auction_synth(17)
        e.step_random(2)
    check_same(t, r, what + ", early starters")
    t.exchange_synth(True); r.exchange_synth(True)
    chains(t, r, DESYNC_CHAIN, what)
    score_both(t, r, ref, what)


def run_external(t, r, mode, gid, ref, what, salt):
    """The oracle's cards from outside, one launch at a time; at every launch a seeded ~1/7 of the live games get
    TAROK_CARD_SKIP and catch up later, so the tiles desynchronise.  A per-game play pointer stays on the device."""
    import tarok_b200.env as E
    n = t.n
    t.reset_stats(); r.reset_stats()
    t.setup_synth(mode, gid); r.setup_synth(mode, gid)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(salt)
    rows = torch.arange(n, device="cuda")
    ptr = torch.zeros(n, dtype=torch.long, device="cuda")
    launches = 0
    while True:
        live = ((t.meta[:n] >> E.M_PHASE) & 3) == E.PH_PLAY
        if not bool(live.any()):
            break
        assert launches < 160, what
        skip = live & (torch.randint(0, 7, (n,), generator=gen, device="cuda") == 0)
        card = ref["cards"][rows, ptr.clamp(max=47)]
        card = torch.where(skip, torch.full_like(card, CARD_SKIP), card).contiguous()
        t.step(card); r.step(card)
        ptr += (live & ~skip).long()
        launches += 1
        check_same(t, r, "%s, launch %d" % (what, launches))
    assert bool((ptr == ref["plays"]).all()), what
    score_both(t, r, ref, what)
    return launches


@pytest.mark.parametrize("case,impl", [(c, i) for c in CASES for i in (2, 3)])
def test_persistent_step_kernel_loops_over_tiles(oracle, tmp_path, case, impl):
    """Impl 2 or 3, PDL on and off, modes 16 / 17 / 0 at an even and an odd first game id, through: the graph-backed
    stepwise rollout; the same with plain launches; setup + random chains of several lengths; the desynchronised mode-17
    batch; and (impl 2) external cards with skips.  Every run against the oracle, every chain / external launch against the
    plain kernel."""
    from tarok_b200.env import TarokEnv
    S = sms()
    n = case_size(case, S)
    t = TarokEnv(n, seed=SEED, history=True)
    r = TarokEnv(n, seed=SEED, history=True)
    r.set_step_impl(1)
    t.set_step_impl(impl)
    traced = set()

    def run(entry, fn, **expect):
        """fn() -- under the profiler, with its play_step launches checked, the first time this entry runs."""
        if entry in traced:
            return fn()
        traced.add(entry)
        box = []
        launches = step_launches(lambda: box.append(fn()), tmp_path / ("%s%d_%s.pt.trace.json" % (case, impl, entry)))
        if entry == "external":                    # as many launches as the skips made necessary, on both handles
            expect.update(total=box[0], plain=box[0])
        check_launches(launches, case, impl, what="case %s impl %d, first %s run" % (case, impl, entry), **expect)
        return box[0]

    try:
        if case == "D":
            if impl == 3:
                # above 3 M deals the draw cache is off by default, and impl 3 then runs the plain kernel throughout
                ref = reference(oracle, n, 16, GIDS[0])
                t.reset_stats()
                run("default_draw_cache", lambda: t.rollout(16, first_game_id=GIDS[0]), total=48, pp=0, graph=False)
                check_oracle(t, ref, "case D impl 3, default draw cache")
            t.set_draw_cache(3)
            force_graph(t)
        graph = impl == 3                          # the stepwise rollout never replays a graph with k_step_tma
        for pdl in (True, False):
            t.set_pdl(pdl)
            for mode in MODES:
                for gid in GIDS:
                    ref = reference(oracle, n, mode, gid)
                    what = "case %s (n = %d) impl %d pdl %d mode %d gid %d" % (case, n, impl, pdl, mode, gid)
                    t.reset_stats()
                    run("rollout", lambda: t.rollout(mode, first_game_id=gid), total=48, pp=pp_launches((48,)), graph=graph)
                    check_oracle(t, ref, what + ", rollout")
                    if impl == 3:                  # (with impl 2 the rollout above already made plain launches)
                        t.set_graph(False)
                        t.reset_stats()
                        run("rollout_plain", lambda: t.rollout(mode, first_game_id=gid), total=48, pp=pp_launches((48,)),
                            graph=False)
                        check_oracle(t, ref, what + ", rollout, plain launches")
                        if case == "D":
                            force_graph(t)
                        else:
                            t.set_graph(True)
                    run("chain", lambda: run_chain(t, r, mode, gid, ref, what + ", chains"), total=sum(CHAIN),
                        plain=sum(CHAIN), pp=pp_launches(CHAIN), graph=False)
                    if mode == 17:
                        k = 2 + sum(DESYNC_CHAIN)
                        run("desync", lambda: run_desync(t, r, gid, ref, what + ", desynchronised"), total=k, plain=k,
                            pp=pp_launches((2,) + DESYNC_CHAIN), graph=False)
                    if impl == 2:
                        run("external", lambda: run_external(t, r, mode, gid, ref, what + ", external cards",
                                                             salt=mode * 2 + (gid & 1)),
                            total=None, pp=0, graph=False, random=False)
        for (c, key), (grid, tiles, iters) in sorted(SEEN.items()):
            if c == case:
                print("case %s, %d SMs: %s grid %d over %d tiles, %d iterations" % (case, S, key, grid, tiles, iters))
    finally:
        t.close()
        r.close()
