"""Timing of the mixed-table entries on one GPU (CUDA events; prints the card and its power limit).

  1. Per-launch time of play_step at 1,048,576 games: tarok_step_bots with seat mask 0, 0x0F and a uniform random mask per
     game, against tarok_step and tarok_step_random.  Every variant plays the SAME games: the deals and contracts of
     setup_synth(18), the cards a step_random chain plays (recorded once), so the fed cards are legal and a bot draws exactly
     the card that was recorded.  Four environments take the launches of a step in turn, so the state a launch touches
     (4 x ~60 MB between two launches on one environment) is not in the 126 MB L2; the variants alternate within one call.
  2. Samoigra section times at 65,536 envs (fp32): boti=() against boti=(2, 3).
usage: python tools/bots_bench.py [--out results.json]"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from tarok_b200.env import MODE_AUCTION_BOT, TarokEnv

N, ENVS, REPS = 1 << 20, 4, 5


def card_info():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as ex:                                   # the number still stands, with the limit unknown
        pl = "unknown (%s)" % ex
    return name, pl


def record_cards(fg):
    env = TarokEnv(N, seed=7, history=True)
    env.setup_synth(MODE_AUCTION_BOT, fg)
    env.step_random(48)
    cards = (env.hist[:, :N] & 63).clone()
    cards[env.hist[:, :N] == 0xFF] = 0xFF
    env.close()
    return cards


def step_times():
    envs = [TarokEnv(N, seed=7) for _ in range(ENVS)]
    fgs = [k * N for k in range(ENVS)]
    cards = [record_cards(fg) for fg in fgs]
    dev = envs[0].torch_device
    masks = {"0": torch.zeros(N, dtype=torch.uint8, device=dev), "0x0F": torch.full((N,), 15, dtype=torch.uint8, device=dev),
             "random": torch.randint(0, 16, (N,), dtype=torch.uint8, device=dev)}
    ff = torch.full((N,), 0xFF, dtype=torch.uint8, device=dev)
    variants = {
        "tarok_step": lambda e, k, t: e.step(cards[k][t]),
        "tarok_step_random": lambda e, k, t: e.step_random(),
        "tarok_step_bots mask 0": lambda e, k, t: e.step(cards[k][t], bots=masks["0"]),
        "tarok_step_bots mask 0x0F": lambda e, k, t: e.step(ff, bots=masks["0x0F"]),
        "tarok_step_bots random mask": lambda e, k, t: e.step(cards[k][t], bots=masks["random"]),
    }
    times = {v: [] for v in variants}
    final = {}
    for rep in range(REPS + 1):                               # rep 0 warms every shape up
        for name, fn in variants.items():
            for e, fg in zip(envs, fgs):
                e.reset_stats()
                e.setup_synth(MODE_AUCTION_BOT, fg)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            for t in range(48):
                for k, e in enumerate(envs):
                    fn(e, k, t)
            b.record()
            torch.cuda.synchronize()
            if rep:
                times[name].append(a.elapsed_time(b) * 1e3 / (48 * ENVS))
            for e in envs:
                e.score()
            final[name] = [e.stats().tolist() for e in envs]
    ref = final["tarok_step_random"]
    for name, st in final.items():                            # the same games whichever entry played them
        assert st == ref, name
    return {name: dict(median_us=float(np.median(v)), min_us=float(np.min(v)), max_us=float(np.max(v)))
            for name, v in times.items()}


def samoigra_sections(n=1 << 16, reps=3):
    from tarok_b200.mreze import ustvari_mreze
    from tarok_b200.samoigra import Samoigra
    torch.manual_seed(1)
    mreze = [ustvari_mreze(torch.device("cuda")) for _ in range(4)]
    runs = {"boti=()": Samoigra(n, mreze=mreze, seed=3), "boti=(2,3)": Samoigra(n, mreze=mreze, seed=3, boti=(2, 3))}
    out = {k: [] for k in runs}
    for rep in range(reps + 1):
        for k, s in runs.items():
            torch.cuda.synchronize()
            t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
            t0.record()
            _, ms = s.odigraj(first_game_id=rep * n, meri=True)
            t1.record()
            torch.cuda.synchronize()
            if rep:
                ms["total (one rollout)"] = t0.elapsed_time(t1)
                out[k].append(ms)
    return {k: {sec: float(np.median([m[sec] for m in v])) for sec in v[0]} for k, v in out.items()}


if __name__ == "__main__":
    path = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    name, pl = card_info()
    res = dict(card=name, power_limit=pl, games=N, envs=ENVS, step_us_per_launch=step_times(),
               samoigra_ms_65536_fp32=samoigra_sections())
    print(json.dumps(res, indent=1))
    if path:
        os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
        with open(path, "w") as f:
            json.dump(res, f, indent=1)
