"""Direct large-N parity GPU -> reference (BASELINE config 1 "exactly": 10,000 Klop deals; 2,000 deals of each other contract).

tests/golden/gpu_traces.npz holds games PLAYED BY THE CUDA KERNELS on a B200 (tools/export_gpu_traces.py): Philox deals,
uniform-random legal-move players, per play the card and a digest of the legal mask the device showed.
* build container (`reference` marker): every game is replayed through the imported, unmodified Python reference -- the
  recorded cards are teacher-forced, the reference's own `mozne` at every play, its trick winners and its scores must equal
  what the GPU produced;
* everywhere (CPU): the same replay through the C oracle;
* GPU box (`gpu` marker): the kernels regenerate the traces from the same seed and must reproduce the committed file array
  for array, which ties the CURRENT kernels to the replayed games.
The file stores the deals, the cards played and the per-game mask digests as one sha256 per 100 games
(tools/export_gpu_traces.py `compact`); the C oracle's synthetic rollout regenerates the deals and the cards from the seed, and
they must match."""
import hashlib
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
PATH = os.path.join(HERE, "golden", "gpu_traces.npz")
pytestmark = pytest.mark.skipif(not os.path.exists(PATH), reason="tests/golden/gpu_traces.npz not generated yet")


def _check_digests(got, want, what):
    """``got``: the array of all games; ``want``: its stored digests.  A mismatch names the first block of games that differs."""
    X = _tool()
    d = X.digests(got)
    assert d.shape == want.shape, (what, d.shape, want.shape)
    bad = np.flatnonzero((d != want).any(1))
    assert not len(bad), "%s differs in games %d..%d" % (what, bad[0] * X.DIGEST_GAMES, (bad[0] + 1) * X.DIGEST_GAMES - 1)


def _tool():
    tools = os.path.join(os.path.dirname(HERE), "tools")
    if tools not in sys.path:
        sys.path.insert(0, tools)
    import export_gpu_traces as X
    return X


@pytest.fixture(scope="module")
def stored():
    return dict(np.load(PATH))


@pytest.fixture(scope="module")
def tr(stored, oracle):
    """The committed games with their deals (`perm`) and cards (`card`) restored and checked against the stored digests."""
    t = dict(stored)
    assert (t["err"] == 0).all()                       # the digests cover every game: none may be an error game
    seed = int(t["seed"][0])
    ends = list(t["first"][1:]) + [len(t["contract"])]
    parts = [oracle.rollout(seed, int(a), int(b - a), int(t["contract"][a])) for a, b in zip(t["first"], ends)]
    t["perm"] = np.concatenate([p["perm"] for p in parts])
    t["card"] = np.concatenate([p["cards"] for p in parts])
    for k in ("perm", "card"):
        _check_digests(t[k], t[k + "_sha256"], k)
    return t


def _digest(masks):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(masks, np.uint64).tobytes()).digest()[:16], np.uint8)


def test_gpu_traces_replay_through_the_c_oracle(tr, oracle):
    n = len(tr["contract"])
    assert n == 28000 and (tr["contract"][:10000] == 0).all()                       # config 1 exactly + 9 x 2,000
    ok = tr["err"] == 0
    rep = oracle.replay(tr["perm"], tr["contract"], tr["declarer"], tr["king"], tr["group"], tr["discard"], tr["card"],
                        want_state=False)
    assert (rep["err"][ok] == 0).all()
    assert (rep["scores"][ok] == tr["scores"][ok]).all()
    assert (rep["plays"][ok] == tr["plays"][ok]).all()
    played = tr["card"] != 0xFF
    assert (rep["seat"][played & ok[:, None]] == tr["seat"][played & ok[:, None]]).all()
    tricks = (tr["plays"] // 4)
    for k in range(12):
        sel = ok & (tricks > k)
        assert (rep["winner"][sel, k] == tr["winner"][sel, k]).all(), k
    masks = np.where(played, rep["mask"], 0).astype(np.uint64)
    dig = np.stack([_digest(masks[i]) for i in range(n)])
    _check_digests(dig, tr["mask_digest_sha256"], "legal masks")
    for c in range(10):                                                              # and the masks stored whole
        a = int(tr["first"][c])
        m = tr["mask_full"][c]
        assert (np.where(played[a:a + len(m)], m, 0) == masks[a:a + len(m)])[ok[a:a + len(m)]].all()


def _replay_chunk(args):
    """Worker: replays games [a, b) (`tr` = their rows) through the reference; returns the mismatching game indices and the
    digest of the legal masks the reference showed in every game."""
    a, b, tr = args
    from oracle import ref_harness as H
    bad, digests = [], []

    class Forced(H.Policy):
        def __init__(self, i):
            super().__init__()
            self.i, self.t = i - a, 0

        def group(self, seat, kupcki):
            return int(tr["group"][self.i])

        def discards(self, seat, mozno, k):
            want = int(tr["discard"][self.i])
            out = [c for c in mozno if (want >> c.v_id()) & 1]
            assert len(out) == k and sum(1 << c.v_id() for c in out) == want
            return out

        def card(self, seat, stih, mozne, zgodovina):
            c = int(tr["card"][self.i][self.t])
            self.t += 1
            return next(k for k in mozne if k.v_id() == c)          # StopIteration = the GPU played a card the reference forbids

    for i in range(a, b):
        j = i - a
        masks = np.zeros(48, np.uint64)
        try:
            rec, players = H.run_forced(tr["perm"][j], int(tr["contract"][j]), int(tr["declarer"][j]), int(tr["king"][j]), Forced(i))
        except Exception as ex:                                     # noqa: BLE001 - any divergence is a failure of this game
            bad.append((i, repr(ex)[:80]))
            digests.append(_digest(masks))
            continue
        p = int(tr["plays"][j])
        masks[:p] = np.array(rec.masks, np.uint64)
        digests.append(_digest(masks))
        good = (len(rec.cards) == p and list(tr["seat"][j][:p]) == rec.seats and list(tr["scores"][j]) == rec.scores
                and list(tr["winner"][j][:p // 4]) == rec.winners)
        if not good:
            bad.append((i, "differs"))
    return bad, digests


@pytest.mark.reference
def test_gpu_traces_replay_through_the_python_reference(tr):
    """Every GPU-played game through the imported anzeA/Tarok engine (per-contract constructors, deal injection)."""
    import multiprocessing as mp
    n = len(tr["contract"])
    workers = min(8, os.cpu_count() or 1)
    step = (n + 8 * workers - 1) // (8 * workers)
    keys = ("perm", "contract", "declarer", "king", "group", "discard", "card", "seat", "scores", "winner", "plays")
    chunks = [(a, min(n, a + step), {k: tr[k][a:a + step] for k in keys}) for a in range(0, n, step)]
    with mp.get_context("spawn").Pool(workers) as pool:
        parts = pool.map(_replay_chunk, chunks)
    bad = [x for part, _ in parts for x in part]
    assert not bad, bad[:5]
    dig = np.stack([d for _, part in parts for d in part])
    _check_digests(dig, tr["mask_digest_sha256"], "legal masks shown by the reference")


@pytest.mark.gpu
def test_current_kernels_regenerate_the_committed_traces(stored, tmp_path):
    X = _tool()
    got = X.export(str(tmp_path / "again.npz"))
    for k in ("contract", "declarer", "king", "group", "discard", "seat", "winner", "scores", "plays", "err", "mask_full"):
        assert np.array_equal(np.asarray(got[k]), stored[k]), k
    for k in X.DIGESTED:
        _check_digests(got[k], stored[k + "_sha256"], k)
