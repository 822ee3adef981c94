"""Observation element type (fp32 / bf16 / fp16) at BASELINE config-4 scale: the kernel and the self-play loop.

    python tools/obs_dtype_bench.py OUT_DIR [--n 65536] [--mode 18] [--reps 5] [--rollouts 3]

Leg 1, the kernel: one rollout of n envs with history (setup of `mode`, then uniform-random plays); at every step
obs_buckets(4), then k_obs_expand_all (tarok_obs_expand_buckets_ex) into fp32, bf16 and fp16 arenas, the dtypes alternated,
`reps` repetitions each, every launch timed with CUDA events.  Reported per dtype: ms per rollout (per-step mean over the
repetitions, summed over the steps), bytes written per rollout computed from the bucket counts, and bytes / time.

Leg 2, self-play: Samoigra.odigraj(meri=True) with the same random-init nets in each dtype, one warm-up rollout each, then
`rollouts` rounds alternating the dtypes; every section (env, bucket, obs, select, forward) per rollout.

Prints the device name and power limit with the numbers and writes OUT_DIR/obs_dtype_bench.json."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from tarok_b200 import env as E  # noqa: E402

DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}
# elements of the per-game vectors k_obs_expand_all writes, by net type (Klop, Navadna_igra, Solo, Berac):
# talon_klop 54 | talon 330 + king 4 + decl 4 + discard 54 | talon 330 + decl 4 + discard 54 | decl 4
VECTOR_ELEMS = np.array([54, 330 + 4 + 4 + 54, 330 + 4 + 54, 4], np.int64)


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.stdout else q.stderr}


def elements_written(cnt):
    """Elements k_obs_expand_all writes for the bucket counts of one step (384 uint32)."""
    total = 0
    for k in range(127):
        size = int(cnt[k])
        if size:
            T, net = 8 * (k % 7 + 1), (k % 28) // 7
            total += size * (T * 216 + int(VECTOR_ELEMS[net]))
    return total


def leg_kernel(n, mode, reps):
    env = E.TarokEnv(n, seed=0x0B5D7, history=True)
    env.setup_synth(mode, 0)
    dev = env.torch_device
    arenas = {name: _arenas(n, dev, dt) for name, dt in DTYPES.items()}
    ms = {name: 0.0 for name in DTYPES}
    elems, steps = 0, 0
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps * len(DTYPES))]
    for t in range(48):
        _, cnt = env.obs_buckets(4)
        total = int(cnt[255])
        if total == 0:
            break
        if t == 0:                                                     # warm-up: first launch of each instantiation
            for name in DTYPES:
                env.obs_expand_buckets(total, *arenas[name])
        slot = {}
        for r in range(reps):
            for j, name in enumerate(DTYPES):
                a, b = ev[r * len(DTYPES) + j]
                a.record()
                env.obs_expand_buckets(total, *arenas[name])
                b.record()
                slot.setdefault(name, []).append((a, b))
        torch.cuda.synchronize()
        for name, pairs in slot.items():
            ms[name] += sum(a.elapsed_time(b) for a, b in pairs) / reps
        elems += elements_written(cnt)
        steps += 1
        env.step_random(1)
    env.close()
    out = {}
    for name, dt in DTYPES.items():
        byts = elems * torch.finfo(dt).bits // 8
        out[name] = {"ms_per_rollout": ms[name], "bytes_written": byts, "GB_per_s": byts / (ms[name] * 1e-3) / 1e9}
    return {"n": n, "mode": mode, "steps": steps, "reps": reps, "dtypes": out}


def _arenas(n, dev, dt):
    from tarok_b200.samoigra import _Arena
    a = _Arena(n, dev, dt)
    return (a.opp, a.hand, a.talon, a.talon_klop, a.king, a.decl, a.disc)


def leg_selfplay(n, rollouts):
    from tarok_b200.mreze import ustvari_mreze
    from tarok_b200.samoigra import Samoigra
    torch.manual_seed(0)
    mreze = [ustvari_mreze(torch.device("cuda", 0)) for _ in range(4)]
    games, out = {}, {}
    for name, dt in DTYPES.items():
        try:
            games[name] = Samoigra(n, mreze=mreze, seed=0x5A1, dtype=dt)
            games[name].odigraj(first_game_id=0)                       # warm-up
            out[name] = {"rollouts": []}
        except Exception as ex:                                        # e.g. a forward the library rejects in this dtype
            out[name] = {"error": "%s: %s" % (type(ex).__name__, str(ex)[:400])}
            games.pop(name, None)
    for r in range(rollouts):
        for name, s in games.items():
            torch.cuda.synchronize()
            st, ms = s.odigraj(first_game_id=1 + r, meri=True)
            ms = {k: round(v, 3) for k, v in ms.items()}
            ms["total_sections"] = round(sum(ms.values()), 3)
            out[name]["rollouts"].append({"ms": ms, "finished": int(st[18]), "error_games": int(st[20])})
    for s in games.values():
        s.zapri()
    return {"n": n, "dtypes": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--n", type=int, default=65536)
    ap.add_argument("--mode", type=int, default=E.MODE_AUCTION_BOT)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rollouts", type=int, default=3)
    ap.add_argument("--legs", default="kernel,selfplay")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("obs_dtype_bench needs a CUDA device")
    os.makedirs(a.out_dir, exist_ok=True)
    res = {"device": device_info()}
    print("device:", res["device"], flush=True)
    if "kernel" in a.legs:
        res["kernel"] = leg_kernel(a.n, a.mode, a.reps)
        for name, d in res["kernel"]["dtypes"].items():
            print("k_obs_expand_all %s: %8.3f ms per rollout, %7.1f MB written, %6.0f GB/s" % (
                name, d["ms_per_rollout"], d["bytes_written"] / 1e6, d["GB_per_s"]), flush=True)
    if "selfplay" in a.legs:
        res["selfplay"] = leg_selfplay(a.n, a.rollouts)
        for name, d in res["selfplay"]["dtypes"].items():
            for r in d.get("rollouts", [d]):
                print("Samoigra %s:" % name, r, flush=True)
    with open(os.path.join(a.out_dir, "obs_dtype_bench.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
