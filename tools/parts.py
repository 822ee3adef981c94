"""CUDA-event timing of the pipeline parts at a given batch size: setup, random steps, forced steps, score, fused.
   python tools/parts.py [games] [mode]      (TAROK_B200_LIB selects a variant build)"""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from tarok_b200.env import TarokEnv


def timed(fn, reps=10):
    fn(); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / reps * 1e3


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 1 << 20
    mode = int(sys.argv[2]) if len(sys.argv) > 2 else 16
    out = {"lib": os.path.basename(os.environ.get("TAROK_B200_LIB", "libtarok_b200.so")), "games": n, "mode": mode}
    rec = TarokEnv(n, seed=1, history=True)
    rec.setup_synth(mode, 0); rec.step_random(48)
    hist = rec.hist
    acts = torch.where(hist == 0xFF, hist, hist & 63).contiguous()
    del hist
    rec.close()
    env = TarokEnv(n, seed=1)
    env.set_materialise(False)
    if os.environ.get("TAROK_DRAW_CACHE"):
        env.set_draw_cache(int(os.environ["TAROK_DRAW_CACHE"]))
        out["draw_cache"] = int(os.environ["TAROK_DRAW_CACHE"])
    if os.environ.get("TAROK_LAZY_MASK") == "0":
        env.set_lazy_mask(False)
        out["lazy_mask"] = 0
    out["setup_us"] = timed(lambda: env.setup_synth(mode, 0))

    def steps(forced):
        env.setup_synth(mode, 0)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        if forced:
            for t in range(48):
                env.step(acts[t])
        else:
            env.step_random(48)
        b.record()
        return a, b
    for name, forced in (("step_random_us", False), ("step_forced_us", True)):
        steps(forced); torch.cuda.synchronize()
        ev = [steps(forced) for _ in range(10)]
        torch.cuda.synchronize()
        out[name] = sum(a.elapsed_time(b) for a, b in ev) / len(ev) / 48 * 1e3
    out["score_us"] = timed(lambda: env.score())
    out["fused_us"] = timed(lambda: env.rollout(mode, 0, fused=True))
    out["stepwise_rollout_us"] = timed(lambda: env.rollout(mode, 0, fused=False))
    env.close()
    print(json.dumps({k: (round(v, 2) if isinstance(v, float) else v) for k, v in out.items()}))


if __name__ == "__main__":
    main()
