"""GPU: the host-buffer entries -- tarok_rollout_host (fused and stepwise), tarok_rollout_records and
tarok_rollout_host_packed -- game by game against the C oracle's rollout of injected deals (oracle.rollout_injected).

The deals are numpy permutations, not Philox deals, so an entry that re-dealt from the game id would fail; the contracts
mix all ten per game.  The game ids include one above 2^32 and the form bench.py uses, so the play draws, the discards and
the player sums (player = (seat + game id) & 3) check that every chunk of the upload / play / download pipeline plays its
games under their own ids.  Bar: bit-exact scores and statistics."""
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SEED = 0x5EED0017
KING_GAMES = (1, 2, 3)
NON_KING = (0, 4, 5, 6, 7, 8, 9)           # Klop, Solo tri/dve/ena, Berac, Solo brez, Odprti berac
ENTRIES = ("rows_fused", "rows_stepwise", "records", "packed1", "packed3", "packed16")


def bench_gid(n):
    """bench.py's game id of a host-entry call: i * total + rank * n, here step i = 3 on rank 1 of 2."""
    return 3 * (2 * n) + 1 * n


GIDS = (0, 2 ** 32 + 12345, "bench")


def chunk_bounds(n, want, quantum=2048):
    """tarok_chunk_bounds (tarok_host.cpp) with the pack pool's block of 2048 rows: the tapered upload chunks."""
    want = min(want, 32)
    if want < 2 or n < (1 << 18):
        return [0, n]
    units = [1 if want < 4 else (1 if e == 0 else 2 if e == 1 else 4) for e in (min(c, want - 1 - c) for c in range(want))]
    bounds, acc = [0], 0
    for c in range(want):
        acc += units[c]
        b = (n * acc // sum(units) + quantum - 1) // quantum * quantum
        if b > n or c == want - 1:
            b = n
        if b > bounds[-1]:
            bounds.append(b)
        if b == n:
            break
    return bounds


@functools.lru_cache(maxsize=2)
def inputs(n, contracts=tuple(range(10)), salt=0):
    """Deals and forced contracts drawn by numpy, independent of any game id: permutation rows, a contract per game from
    `contracts`, a uniform declarer, a uniform king for Tri/Dve/Ena and 7 (none) otherwise."""
    rng = np.random.default_rng([n, salt])
    perm = rng.permuted(np.tile(np.arange(54, dtype=np.uint8), (n, 1)), axis=1)
    contract = np.asarray(contracts, np.uint8)[rng.integers(0, len(contracts), n)]
    declarer = rng.integers(0, 4, n, dtype=np.uint8)
    king = np.where(np.isin(contract, KING_GAMES), rng.integers(0, 4, n, dtype=np.uint8), np.uint8(7)).astype(np.uint8)
    return dict(perm=perm, contract=contract, declarer=declarer, king=king)


@functools.lru_cache(maxsize=2)
def reference(n, gid):
    from oracle import oracle as O
    x = inputs(n)
    return O.rollout_injected(SEED, gid, x["perm"], x["contract"], x["declarer"], x["king"])


def pinned(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()


def run(env, entry, x, gid, pin=True, with_king=True, wait=True):
    """One host-entry call on the current stream.  Returns the (scores, stats) host buffers (numpy when pin=False) and the
    input buffers, which must outlive the call's copies when it is not waited for."""
    import torch
    from tarok_b200.env import pack_records
    n = env.n
    if pin:
        ins = {k: pinned(v) for k, v in x.items()}
        scores, stats = torch.empty((n, 4), dtype=torch.int16).pin_memory(), torch.zeros(32, dtype=torch.int64).pin_memory()
    else:
        ins = x
        scores, stats = np.empty((n, 4), np.int16), np.zeros(32, np.int64)
    king = ins["king"] if with_king else None
    if entry == "records":
        ins = dict(ins, records=pack_records(ins["perm"], ins["contract"], ins["declarer"], king)[0])
        env.rollout_records(ins["records"], scores, stats, first_game_id=gid)
    elif entry.startswith("packed"):
        env.rollout_host_packed(ins["perm"], ins["contract"], ins["declarer"], king, scores, stats, first_game_id=gid,
                                threads=int(entry[len("packed"):]))
    else:
        env.rollout_host(ins["perm"], ins["contract"], ins["declarer"], king, scores, stats, first_game_id=gid,
                         fused=entry == "rows_fused")
    if wait:
        torch.cuda.current_stream().synchronize()
    return scores, stats, ins


def np_of(a):
    return a.numpy() if hasattr(a, "numpy") else a


def assert_matches(scores, stats, ref, what):
    from oracle import oracle as O
    sc = np_of(scores)
    bad = np.flatnonzero((sc != ref["scores"]).any(axis=1))
    assert bad.size == 0, "%s: %d games differ from the oracle, first %s" % (what, bad.size, bad[:8].tolist())
    st = np_of(stats)[:21]
    assert (st == O.device_stats(ref)).all(), "%s: stats %s != oracle %s" % (what, st.tolist(), O.device_stats(ref).tolist())


def _env(n, **kw):
    from tarok_b200.env import TarokEnv
    return TarokEnv(n, seed=SEED, **kw)


SIZES = (1, 3, 513, 262_143, 262_144, 300_001, 1_048_577)      # the first four run as one chunk, the rest as several


@pytest.mark.parametrize("n,gid,entry", [(n, g, e) for n in SIZES for g in GIDS for e in ENTRIES],
                         ids=lambda v: str(v))
def test_host_entry_matches_oracle(n, gid, entry):
    gid = bench_gid(n) if gid == "bench" else gid
    env = _env(n)
    scores, stats, _ = run(env, entry, inputs(n), gid)
    env.close()
    assert_matches(scores, stats, reference(n, gid), entry)


@pytest.mark.parametrize("chunks", [1, 2, 3, 8, 32])
@pytest.mark.parametrize("n", [262_145, 1_048_577])
def test_pipeline_depth_does_not_change_a_game(n, chunks):
    """Every pipeline depth (TAROK_OPT_CHUNKS, 1..32 tapered chunks on multiples of 2048 rows) plays the same games."""
    gid = 2 ** 32 + 1
    ref = reference(n, gid)
    env = _env(n)
    env.set_chunks(chunks)
    for entry in ("rows_fused", "records", "packed3"):
        scores, stats, _ = run(env, entry, inputs(n), gid)
        assert_matches(scores, stats, ref, "%s, %d chunks" % (entry, chunks))
    env.close()


def test_king_may_be_null_for_non_king_games():
    """``king = NULL`` (documented for non-king games) through every entry equals an explicit king 7, and the oracle."""
    from oracle import oracle as O
    n, gid = 300_001, 2 ** 33 + 3
    x = inputs(n, NON_KING, salt=1)
    assert (x["king"] == 7).all()
    ref = O.rollout_injected(SEED, gid, x["perm"], x["contract"], x["declarer"], None)
    env = _env(n)
    for entry in ENTRIES:
        a = run(env, entry, x, gid, with_king=False)
        assert_matches(a[0], a[1], ref, entry + ", king=None")
        b = run(env, entry, x, gid, with_king=True)
        assert (np_of(a[0]) == np_of(b[0])).all() and (np_of(a[1]) == np_of(b[1])).all(), entry
    env.close()


def test_invalid_rows_across_chunk_boundaries():
    """Invalid rows (a duplicate card, card id 54, declarer 4) at the first and last row and on both sides of the first two
    chunk bounds: error games with zero scores, counted in stats[20]; every other game as the oracle plays it."""
    from oracle import oracle as O
    n, gid = 1_048_577, 2 ** 32 + 99
    x = {k: v.copy() for k, v in inputs(n).items()}
    b = chunk_bounds(n, 8)
    rows = sorted({0, n - 1, b[1] - 1, b[1], b[2] - 1, b[2]})
    assert len(rows) == 6
    for j, r in enumerate(rows):
        kind = j % 3
        if kind == 0:
            x["perm"][r, 5] = x["perm"][r, 40]                        # a card twice, another one missing
        elif kind == 1:
            x["perm"][r, 50] = 54                                     # no such card
        else:
            x["declarer"][r] = 4                                      # no such seat
    ref = O.rollout_injected(SEED, gid, x["perm"], x["contract"], x["declarer"], x["king"])
    assert ref["err"][rows].all() and (ref["scores"][rows] == 0).all()
    env = _env(n)
    for entry in ("rows_fused", "records", "packed3"):
        scores, stats, _ = run(env, entry, x, gid)
        sc, st = np_of(scores), np_of(stats)
        assert (sc[rows] == 0).all(), entry
        assert st[20] == ref["stats"][9] and st[20] >= len(rows), entry
        assert_matches(sc, st, ref, entry)
    env.close()


def test_calls_in_flight_on_one_handle():
    """Three calls on one handle on a side stream with no host synchronisation between them -- rows fused, packed with a
    new thread count (the pool is rebuilt), records -- each with its own inputs, game ids and pinned outputs.  Only the
    side stream is synchronised; each output is its own call's, and each stats vector holds its own call's games only."""
    import torch
    from oracle import oracle as O
    n = 300_001
    calls = [("rows_fused", 0, 2 ** 32 + 5), ("packed16", 1, bench_gid(n)), ("records", 2, 77)]
    env = _env(n)
    run(env, "packed3", inputs(n, salt=9), 0)                        # a pool of 3 threads, so packed16 rebuilds it
    side = torch.cuda.Stream()
    outs = []
    with torch.cuda.stream(side):
        for entry, salt, gid in calls:
            x = inputs(n, salt=10 + salt)
            outs.append(run(env, entry, x, gid, wait=False) + (x,))
    side.synchronize()
    for (entry, salt, gid), (scores, stats, _, x) in zip(calls, outs):
        ref = O.rollout_injected(SEED, gid, x["perm"], x["contract"], x["declarer"], x["king"])
        assert_matches(scores, stats, ref, entry + " in flight")
    env.close()


def test_pageable_buffers_equal_pinned():
    """Plain numpy inputs and outputs (pageable: the copies complete before the call returns) give the pinned result."""
    n, gid = 300_001, bench_gid(300_001)
    ref = reference(n, gid)
    env = _env(n)
    for entry in ("rows_fused", "packed3"):
        p = run(env, entry, inputs(n), gid)
        q = run(env, entry, inputs(n), gid, pin=False)
        assert isinstance(q[0], np.ndarray)
        assert (np_of(p[0]) == q[0]).all() and (np_of(p[1]) == q[1]).all(), entry
        assert_matches(q[0], q[1], ref, entry + ", pageable")
    env.close()
