"""Exports GPU-played games for the direct GPU -> reference replay (tests/test_gpu_traces_vs_reference.py):

    python tools/export_gpu_traces.py gpurun_out/gpu_traces.npz          (on the GPU box, under gpurun)

BASELINE config 1 exactly -- 10,000 Philox Klop deals, four uniform-random legal-move players -- plus 2,000 deals of each
other contract (forced per game, uniform declarer / king, Bot-style exchange), all played by the stepwise CUDA kernels.
Per game: the deal as the permutation Igra.razdeli would have consumed, contract / declarer / king, talon group and
discards, the 48 cards with their seats, a digest of the 48 legal masks the device showed (full masks for the first games of
every contract), trick winners, scores.  The committed copy is tests/golden/gpu_traces.npz, written in the form ``compact``
gives; the tests replay every game through the C oracle (and the imported Python reference where it is installed), the GPU
test regenerates the file and compares it array for array."""
import hashlib
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

SEED = 0xC0FFEE2026
PLAN = [(0, 10000)] + [(c, 2000) for c in range(1, 10)]        # (contract code, deals)
FULL_MASKS = 64                                                # games per contract whose 48 masks are stored whole
# stored as sha256 digests, which keeps the committed file small: the deals and the cards played are regenerated from the
# seed by the C oracle's synthetic rollout, the per-game mask digests by its replay
DIGESTED = ("perm", "card", "mask_digest")
DIGEST_GAMES = 100                                             # games per digest, so that a mismatch names its games


def mask_digest(masks_row):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(masks_row).tobytes()).digest()[:16], np.uint8)


def digests(a):
    """sha256 of every DIGEST_GAMES consecutive games (rows of ``a``): uint8 [ceil(n / DIGEST_GAMES), 32]."""
    a = np.ascontiguousarray(a)
    return np.stack([np.frombuffer(hashlib.sha256(a[i:i + DIGEST_GAMES].tobytes()).digest(), np.uint8)
                     for i in range(0, len(a), DIGEST_GAMES)])


def compact(out):
    """The stored form of ``export``'s arrays: every DIGESTED array ``k`` becomes ``k_sha256`` (``digests``)."""
    c = {k: v for k, v in out.items() if k not in DIGESTED}
    c.update({k + "_sha256": digests(out[k]) for k in DIGESTED})
    return c


def play(contract, n, gid0):
    import torch
    import tarok_b200.env as E
    u64 = lambda t: t.cpu().numpy().view(np.uint64)
    env = E.TarokEnv(n, seed=SEED, history=True)
    env.deal(gid0)
    perm = env.export_perm().cpu().numpy()
    env.force_contract_synth(contract)
    env.exchange_synth(False)
    m = u64(env.meta[:n]).copy()
    f = lambda sh, b: ((m >> np.uint64(sh)) & np.uint64((1 << b) - 1)).astype(np.uint8)
    out = dict(perm=perm, contract=f(E.M_CONTRACT, 4), declarer=f(E.M_DECL, 2), king=f(E.M_KING, 3), group=f(E.M_GROUP, 3),
               discard=u64(env.discard[:n]).copy())
    out["group"] = np.where(out["group"] == 7, 0xFF, out["group"]).astype(np.uint8)
    masks = np.zeros((n, 48), np.uint64)
    for t in range(48):
        masks[:, t] = u64(env.mask[:n])
        env.step_random()
    sc = env.score().cpu().numpy().copy()
    hist = env.hist[:, :n].cpu().numpy().T
    m = u64(env.meta[:n]).copy()
    plays = f(E.M_PLAYS, 6)
    last = f(E.M_WINNER, 2)
    assert int(f(E.M_ERR, 1).sum()) == 0 or contract in (1, 2, 3, 4, 5, 6)
    seat = np.where(hist == 0xFF, 0xFF, hist >> 6).astype(np.uint8)
    card = np.where(hist == 0xFF, 0xFF, hist & 63).astype(np.uint8)
    winner = np.full((n, 12), 0xFF, np.uint8)
    for k in range(12):
        done = plays >= 4 * (k + 1)
        nxt = plays >= 4 * (k + 1) + 1
        if k < 11:
            winner[nxt, k] = seat[nxt, 4 * (k + 1)]                       # the winner leads the next trick
        fin = done & ~nxt
        winner[fin, k] = last[fin]                                        # the final trick: meta's last-winner field
    out.update(seat=seat, card=card, winner=winner, scores=sc.astype(np.int16), plays=plays, err=f(E.M_ERR, 1),
               mask_digest=np.stack([mask_digest(masks[i]) for i in range(n)]), mask_full=masks[:FULL_MASKS].copy())
    env.close()
    return out


def export(path):
    parts, gid0 = [], 0
    for contract, n in PLAN:
        parts.append(play(contract, n, gid0))
        gid0 += n
    out = {k: np.concatenate([p[k] for p in parts]) for k in parts[0] if k != "mask_full"}
    out["mask_full"] = np.stack([p["mask_full"] for p in parts])          # [10, FULL_MASKS, 48]
    out["first"] = np.cumsum([0] + [n for _, n in PLAN])[:-1].astype(np.int64)
    out["seed"] = np.array([SEED], np.uint64)
    np.savez_compressed(path, **compact(out))
    return out


if __name__ == "__main__":
    p = sys.argv[1] if len(sys.argv) > 1 else "gpurun_out/gpu_traces.npz"
    o = export(p)
    print(p, len(o["contract"]), "games", os.path.getsize(p), "bytes; errors", int(o["err"].sum()))
