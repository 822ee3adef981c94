#!/usr/bin/env python
"""bench.py -- env-steps/s and deals/s of the batched Tarok environment (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--games G] [--mode M] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch: deal -> contract -> talon exchange ->
48 x play_step (uniform-random legal-move players) -> score, for G concurrent deals per GPU
(default: BASELINE config 2 = 1,048,576 Navadna deals on one B200).  Prints ONE JSON line.

* value        whole-job env-steps/s, inputs resident in HBM (Philox deals generated on device); each of the K steps
               is bracketed by its own CUDA-event pair, a 160 MiB L2-flush write runs between the pairs
* e2e          same metric through the host-buffer C-ABI entry: pinned host permutation rows + contracts uploaded, scores +
               stats downloaded, inside the timed region; the fastest COMPLETE pipeline from rows is the headline
               (raw 57-byte rows, or rows serialised into 20-byte records by host threads inside the call)
* roofline     the dominant kernel k_step<random>: 64 B/env-step (SURVEY.md 8d) x live games per launch / its CUDA-event
               duration over the timed region, against MEASURED_PEAKS.json; `traffic` = ncu dram bytes per launch
* step_forced  the same 48 steps driven by a device-resident action buffer (k_step<false>: what an external policy uses)
* config3/4/5  BASELINE's other configurations as sub-records (sharded over the ranks; stats_sha256 of the all-reduced
               statistics -- through the C-ABI collective tarok_allreduce_stats -- is identical at every GPU count)
* cpu_baseline the C port of the reference rules (oracle/, OpenMP over all host cores) on a bounded sample of the same
               workload, and -- where the Python reference exists on the box -- the reference itself
* --impl reference  times that same CPU port as the reference arm
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SEED = 0x5EED7A20C0001
BYTES_PER_ENV_STEP = 64          # SURVEY.md 8(d): play_step with the mask fused in
MODE_NAMES = {16: "Navadna igra (Tri/Dve/Ena forced, uniform declarer+king), talon exchange",
              17: "uniform index2igra bids (all contracts incl. Berac), random talon group",
              18: "Bot_igralec bidding (Klop/Tri/Dve/Ena)", 0: "Klop forced"}
CONFIG3_TOTAL = 4_194_304        # BASELINE config 3: 4M concurrent deals over the box
CONFIG5_TOTAL = 16_777_216       # BASELINE config 5: 16M concurrent deals at 1/2/4/8 GPUs
CONFIG4_ENVS = 65_536            # BASELINE config 4: envs per GPU
DUMP_BYTES = 64 << 20            # --dump-outputs: at most this much over all ranks


def workload_name(mode, games):
    return ("config 2: %s; 4 uniform-random legal-move players; %d concurrent deals per GPU; one step = deal, contract, "
            "talon exchange (one fused setup launch), 48 x play_step, score" % (MODE_NAMES.get(mode, str(mode)), games))


def config_of(args):
    """Identical in both arms (the driver compares them)."""
    return {"workload": workload_name(args.mode, args.games), "games_per_gpu": args.games, "mode": args.mode, "seed": hex(SEED)}


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def dump_outputs(out_dir, rank, world, scores, stats):
    """--dump-outputs: what the timed rollout hands its caller after the last timed step -- that step's per-deal scores by
    seat, and the statistics vector, which accumulates over the K timed steps (reset before the first) and is all-reduced over
    the ranks -- as float .npy files, so that two builds run with the same arguments can be compared output for output.
    Scores beyond this rank's share of DUMP_BYTES are a fixed, seeded sample of deals; `scores_rows` holds their indices in
    the batch."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    name = "scores" if world == 1 else "scores_rank%d" % rank
    rows = (DUMP_BYTES // world - 4096) // (4 * 4 + 8)                   # float32 x4 per deal + its float64 index
    if len(scores) > rows:
        idx = np.sort(np.random.default_rng(SEED).choice(len(scores), rows, replace=False))
        scores = scores[idx]
        np.save(os.path.join(out_dir, name + "_rows.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, name + ".npy"), scores.astype(np.float32))
    if rank == 0:
        np.save(os.path.join(out_dir, "stats.npy"), stats.astype(np.float64))


def step_traffic(games, mode, kernel="k_step<random>"):
    """ncu dram__bytes_read.sum + dram__bytes_write.sum per launch for this batch size, if a capture is committed."""
    try:
        for e in json.load(open(os.path.join(ROOT, "profiles", "step_traffic.json")))["entries"]:
            if int(e["games"]) == games and int(e.get("mode", 16)) == mode and e.get("kernel", "k_step<random>") == kernel:
                return e["dram_bytes_per_launch"]
    except Exception:
        pass
    return None


class ClockSampler:
    """Samples SM clocks / throttle reasons (NVML polling thread, else nvidia-smi) while the timed legs run."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None
        self.nvml, self.samples, self.stop_flag = None, [], False

    def _nvml_loop(self):
        import pynvml as N
        h = N.nvmlDeviceGetHandleByIndex(self.index)
        self.mx = N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
        while not self.stop_flag:
            try:
                sm = N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)
                rs = N.nvmlDeviceGetCurrentClocksEventReasons(h)
                self.samples.append((sm, self.mx, rs))
            except Exception:
                break
            time.sleep(0.05)           # 20 Hz: NVML queries share the driver with the CUDA calls of the e2e legs

    def _nvml_result(self):
        import pynvml as N
        self.stop_flag = True
        self.t.join(timeout=2)
        names = {"hw_slowdown": N.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": N.nvmlClocksEventReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": N.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": N.nvmlClocksEventReasonSwPowerCap}
        reasons = sorted(k for k, bit in names.items() if any(s[2] & bit for s in self.samples))
        sm = [s[0] for s in self.samples]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(s[1] for s in self.samples) if sm else None,
                "sm_mhz_min": min(sm) if sm else None, "samples": len(sm), "reasons": reasons,
                "source": "NVML polling thread over every timed GPU leg of this run (headline loop, forced-action leg, e2e legs)"}

    def start(self):
        try:
            import pynvml as N
            N.nvmlInit()
            self.nvml = N
            self.t = threading.Thread(target=self._nvml_loop, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            return self._nvml_result()
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v == "Active":
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------------------------------
# CPU legs (the only places that execute oracle/)
# ----------------------------------------------------------------------------------------------------------------------
def cpu_port_rate(mode, target_seconds):
    """Times the C port of the reference engine (oracle/synth.c, OpenMP) on a bounded sample."""
    from oracle import oracle as O
    O.build()
    cores = O.use_all_threads()
    t = time.perf_counter()
    st = O.rollout_stats_only(SEED, 0, 20000, mode)
    dt = max(time.perf_counter() - t, 1e-4)
    n = int(min(max(20000 / dt * target_seconds, 20000), 40_000_000))
    t = time.perf_counter()
    st = O.rollout_stats_only(SEED, 0, n, mode)
    dt = time.perf_counter() - t
    out = {"steps_per_s": float(st[8]) / dt, "deals_per_s": n / dt, "cores": cores, "deals": n, "seconds": dt}
    O.set_threads(1)                                   # P = 1 beside P = all (BASELINE.md section 3)
    n1 = max(int(n / dt / cores * 2.0), 10000)
    t = time.perf_counter()
    st1 = O.rollout_stats_only(SEED, 0, n1, mode)
    dt1 = time.perf_counter() - t
    O.use_all_threads()
    out["single_core_steps_per_s"] = float(st1[8]) / dt1
    return out


def python_reference_same_box(budget_seconds):
    """The unmodified Python reference timed on THIS box's host cores in THIS run -- possible only where its tree exists
    (/root/reference in the build container, or a tree named by TAROK_REFERENCE_DIR; a Python reference does not travel to the
    GPU box and its sources are not copied into this repository)."""
    try:
        from oracle import ref_harness as H
        if not H.reference_available():
            return {"status": "absent on this box", "looked_in": ["baseline/_ref", "/root/reference"],
                    "container_measurement": "profiles/r02/reference_cpu_container.json (same script, build container)"}
        from oracle import time_reference as TR
        cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        rows = TR.bounded(cores, budget_seconds)
        return {"status": "measured in this run", "tree": H.REFERENCE_DIR, "cores": cores, "python": sys.version.split()[0],
                "players": "4 x Bot_igralec (uniform-random legal moves)", "rows": [
                    {k: r[k] for k in ("workload", "processes", "deals", "env_steps", "seconds", "deals_per_sec", "env_steps_per_sec")}
                    for r in rows]}
    except Exception as ex:
        return {"status": "failed: %s" % str(ex)[:200]}


PY_WORKLOAD_OF_MODE = {16: "navadna_mix", 17: "paralel_start", 18: "paralel_start", 0: "klop", 1: "tri", 2: "dve", 3: "ena",
                       7: "berac", 9: "berac"}


def port_arm(args, seconds_per_step, steps, warmup):
    """The C port of the reference rule engine (oracle/tarok_oracle.c + synth.c, OpenMP, all host threads) on bounded samples."""
    from oracle import oracle as O
    O.build()
    cores = O.use_all_threads()          # torchrun exports OMP_NUM_THREADS=1; the arm uses every host core
    t = time.perf_counter()
    O.rollout_stats_only(SEED, 0, 20000, args.mode)
    rate = 20000 / max(time.perf_counter() - t, 1e-4)
    per_step = int(min(max(rate * seconds_per_step, 20000), args.games))
    for i in range(warmup):
        O.rollout_stats_only(SEED, i * per_step, per_step, args.mode)
    t0 = time.perf_counter()
    env_steps = 0
    for i in range(steps):
        st = O.rollout_stats_only(SEED, (warmup + i) * per_step, per_step, args.mode)
        env_steps += int(st[8])
    dt = time.perf_counter() - t0
    return {"value": env_steps / dt, "unit": "env-steps/s", "cores": cores, "kind": "port", "deals_per_sec": per_step * steps / dt,
            "ms_per_step": dt / steps * 1e3,
            "sample": "%d deals per step (of the %d-deal workload), %d steps" % (per_step, args.games, steps)}


def run_reference(args, rank):
    """Reference arm.  Where the unmodified Python reference is on the box (/root/reference in the build container, or
    TAROK_REFERENCE_DIR) THAT is what is timed -- the same workload through its own classes (Igra.razdeli, Navadna_igra / Klop /
    Berac / Tarok.paralel_start with four Bot_igralec), one process per host core, each step a bounded sample -- and the C port
    of the engine is reported beside it; on the GPU box, where the Python tree cannot be, the C port is the arm."""
    if rank != 0:
        return
    from oracle import ref_harness as H
    use_py = H.reference_available() and not args.no_pyref and args.mode in PY_WORKLOAD_OF_MODE
    if use_py:
        try:
            line = python_arm(args, H)
        except Exception as ex:                                              # anything wrong with the tree or the pool: the port
            print("bench.py: Python reference arm failed (%s); timing the C port instead" % str(ex)[:200], file=sys.stderr)
            line = None
        if line is not None:
            print(json.dumps(line))
            return
    base = port_arm(args, 1.0, args.steps, args.warmup)
    base["python_reference_same_box"] = python_reference_same_box(30.0) if not args.no_pyref else {"status": "skipped (--no-pyref)"}
    v, ms, dps = base["value"], base.pop("ms_per_step"), base["deals_per_sec"]
    note = ("C port of the reference rule engine (oracle/tarok_oracle.c + synth.c, OpenMP): the Python reference is not on this "
            "box; where its tree exists (build container) the same command times the Python engine itself")
    print(json.dumps(reference_line(args, v, ms, dps, base, note)))


def reference_line(args, v, ms, dps, base, note):
    return {"impl": "reference", "metric": "env_steps_per_sec", "value": v, "unit": "env-steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": config_of(args),
            "deals_per_sec": dps,
            "cpu_baseline": base,
            "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": note}


def python_arm(args, H):
    if True:
        from oracle import time_reference as TR
        cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        fn = PY_WORKLOAD_OF_MODE[args.mode]
        H.load_reference()                                                   # once, before the pools fork
        TR.run_workload(fn, 10 * cores, cores)                               # imports, page faults
        probe = TR.run_workload(fn, 60 * cores, cores)
        # a step = about one second of the box's cores (the whole run must end within minutes whatever --steps is)
        budget = min(1.0, 150.0 / max(1, args.steps + args.warmup))
        per_step = max(cores * 8, int(probe["deals_per_sec"] * budget))
        for i in range(args.warmup):
            TR.run_workload(fn, per_step, cores, seed0=1000 + 64 * i)
        env_steps, deals, busy = 0, 0, 0.0
        for i in range(args.steps):
            r = TR.run_workload(fn, per_step, cores, seed0=100000 + 64 * i)
            env_steps += r["env_steps"]; deals += r["deals"]; busy += r["seconds"]
        v = env_steps / busy
        port = port_arm(args, 0.5, 3, 1)
        one = TR.run_workload(fn, max(40, int(probe["deals_per_sec"] / cores * 1.0)), 1)
        base = {"value": v, "unit": "env-steps/s", "cores": cores, "kind": "reference",
                "sample": "%d deals per step through the unmodified Python engine (%s, 4 x Bot_igralec), %d processes, %d steps; a "
                          "step's time = its slowest process (process-pool start-up excluded)" % (per_step, fn, cores, args.steps),
                "tree": H.REFERENCE_DIR, "python": sys.version.split()[0], "single_core_value": one["env_steps_per_sec"],
                "c_port": port}
        ms = busy / args.steps * 1e3
        note = ("the UNMODIFIED Python reference (%s) on every host core; cpu_baseline.c_port = the C restatement of its " % H.REFERENCE_DIR +
                "engine (OpenMP) on the same cores, the conservative comparison")
        return reference_line(args, v, ms, deals / busy, base, note)


# ----------------------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    # libnccl prints its version banner on stdout when NCCL_DEBUG asks for it: everything this process (and the libraries
    # it loads) writes to fd 1 goes to stderr, the ONE JSON line is written to the real stdout at the end
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    import numpy as np
    import torch
    import torch.distributed as dist

    from tarok_b200.dist import NcclComm, shard
    from tarok_b200.env import TarokEnv, pack_records, RECORD_BYTES, MODE_AUCTION_UNIFORM, S_STEPS, S_FINISHED, S_ERRORS

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        from tarok_b200.dist import bind_to_gpu_numa
        bind_to_gpu_numa(local_rank)              # pinned e2e buffers on the GPU's NUMA node
        dist.init_process_group("nccl", device_id=dev)
    n, mode, total = args.games, args.mode, args.games * world
    env = TarokEnv(n, seed=SEED, device=local_rank)
    env.set_materialise(False)      # the rollout's outputs are scores + statistics (Tarok.rezultati); piles stay in the trick log
    comm = NcclComm(local_rank)     # raw ncclComm_t for the C-ABI collective (a one-rank communicator at N = 1)
    auction = mode in (17, 18)
    flush = torch.empty(160 << 20, dtype=torch.uint8, device=dev)          # > 126 MB L2
    stats_ring = torch.zeros((args.warmup + args.steps + 1, 32), dtype=torch.int64, device=dev)
    pending, step_events, iter_events, probe_events = [], [], [], []

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        t = torch.tensor([x], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(t)
        return int(t.item())

    def rollout(i, timed, last=False, probe=False):
        """One step.  Headline form: tarok_rollout_stepwise = ONE graph replay of setup + 48 x play_step + score (51 kernels).
        probe=True: the same kernels as plain launches with a CUDA-event pair around the 48 play_steps (events cannot be
        placed inside a replayed graph) -- used for the roofline's per-launch time, not for `value`."""
        gid0 = i * total + rank * n
        if not args.no_flush:
            flush.zero_()                                                  # L2 flush between iterations (not timed)
        i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        i0.record()
        if probe:
            env.setup_synth(mode, gid0)                                    # deal + contract + exchange, one launch
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            env.step_random(48)
            b.record()
            env.score()
            step_events.append((a, b))
        else:
            env.rollout(mode, first_game_id=gid0, fused=False)
        stats_ring[i % len(stats_ring)].copy_(env.stats_dev)
        if world > 1 and not probe and not os.environ.get("TAROK_BENCH_NO_ALLREDUCE"):   # (diagnostic switch; never set by default)
            # the one collective: returns/statistics, 256 B over NCCL/NVLink; asynchronous so that the next
            # rollout's deal overlaps it (waited for before the timed region closes)
            pending.append(dist.all_reduce(stats_ring[i % len(stats_ring)], async_op=True))
        if last:
            for w in pending:                                              # every all-reduce lands inside a timed interval
                w.wait()
        i1.record()
        if timed:
            (probe_events if probe else iter_events).append((i0, i1))

    for i in range(args.warmup):
        rollout(i, False)
    # the C-ABI collective (tarok_allreduce_stats: raw ncclAllReduce on the handle's vector) against torch.distributed,
    # at every GPU count -- outside the timed region
    via_abi = comm.allreduce_stats(env).cpu().numpy()
    via_torch = env.stats_dev.clone()
    if world > 1:
        dist.all_reduce(via_torch)
    abi_collective_ok = bool((via_abi == via_torch.cpu().numpy()).all())
    assert abi_collective_ok, "tarok_allreduce_stats disagrees with torch.distributed.all_reduce"
    barrier()
    env.reset_stats()
    sampler = ClockSampler(local_rank) if rank == 0 and not os.environ.get("TAROK_BENCH_NO_SAMPLER") else None
    if sampler:
        sampler.start()
    launches0 = env.launches
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if world > 1:
        # device-side start gate: the host barrier lets the ranks go up to a millisecond or two apart (scheduler jitter), and a
        # rank that starts late makes every other rank wait that long for its all-reduces inside their last timed interval.
        # A collective enqueued on the launching stream holds every GPU until all have arrived, so the K steps start together.
        gate = torch.zeros(1, device=dev)
        dist.all_reduce(gate)
    t0.record()
    for i in range(args.steps):
        rollout(args.warmup + i, True, last=(i == args.steps - 1))
    t1.record()
    barrier()
    # K steps, each timed by its own CUDA-event pair on the launching stream (the L2-flush writes run between the pairs)
    region_ms = t0.elapsed_time(t1)
    ms = max_over_ranks(sum(x.elapsed_time(y) for x, y in iter_events))
    st = stats_ring[(args.warmup + args.steps - 1) % len(stats_ring)].cpu().numpy()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, rank, world, env.scores[:n].cpu().numpy(), st)
    launches = env.launches - launches0
    # the same K steps once more as plain launches with an event pair around the 48 play_steps: the roofline's launch time
    probe_stats = env.stats_dev.clone()
    for i in range(args.steps):
        rollout(args.warmup + i, True, probe=True)
    barrier()
    step_ms = max_over_ranks(sum(a.elapsed_time(b) for a, b in step_events) / (48 * len(step_events)))
    probe_ms = max_over_ranks(sum(x.elapsed_time(y) for x, y in probe_events))
    assert bool((env.stats_dev - probe_stats == probe_stats).all()), "the plain-launch pass must repeat the graph pass exactly"
    env_steps, deals, errors = int(st[S_STEPS]), int(st[S_FINISHED]), int(st[S_ERRORS])
    value = env_steps / (ms * 1e-3)

    # ---- roofline of the dominant kernel (k_step<random>) over the timed region
    peak, peak_src = hbm_peak()
    live_per_launch = env_steps / world / (48 * args.steps)               # live games one launch advances
    achieved = BYTES_PER_ENV_STEP * live_per_launch / (step_ms * 1e-3) / 1e9
    traffic = step_traffic(n, mode)
    roofline = {"bound": "hbm", "kernel": "k_step<random>", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "achieved_kind": "ALGORITHMIC bytes (SURVEY 8d: 64 B/env-step) / event-timed launch -- not a measured DRAM rate",
                "algorithmic_bytes_per_launch": BYTES_PER_ENV_STEP * live_per_launch,
                "dram_gbs_from_traffic": (traffic / (step_ms * 1e-3) / 1e9) if traffic else None,
                "dram_frac_from_traffic": (traffic / (step_ms * 1e-3) / 1e9 / peak) if traffic else None,
                "avg_launch_us": step_ms * 1e3,
                "step_kernel_share_of_rollout": step_ms * 48 * args.steps / probe_ms,
                "launch_time_from": "a second pass over the same K steps as plain launches (%.4f ms per step) with a CUDA-event pair "
                                    "around the 48 play_steps; the headline pass replays the same kernels as one CUDA graph per step"
                                    % (probe_ms / args.steps),
                "note": "frac can exceed 1: the kernel moves fewer DRAM bytes than SURVEY's accounting (`traffic`, ncu) and at this "
                        "batch size its 50 MB step working set stays in the 126 MB L2 between launches; dram_frac_from_traffic is the "
                        "physical DRAM rate (ncu bytes / event-timed launch); roofline_large is the same kernel on a state 8x larger than L2"}

    # ---- the same 48 steps with externally supplied actions (k_step<false>: the variant a policy drives) --------------
    forced = None
    if not args.no_forced:
        eh = TarokEnv(n, seed=SEED, device=local_rank, history=True)
        gidf = rank * n
        eh.setup_synth(mode, gidf)
        eh.step_random(48)
        eh.score()
        want_scores = eh.scores[:n].clone()
        hist = eh.hist                                                     # [48, n_alloc] seat << 6 | card, 0xFF = no play
        acts = torch.where(hist == 0xFF, hist, hist & 63).contiguous()     # device-resident action buffer (teacher forcing)
        del hist
        eh.close()
        reps = max(3, min(args.steps, 20))
        ev = []
        # the 48 per-card calls are captured once into a CUDA graph (every entry point only enqueues stream-ordered work): a
        # policy loop written in Python costs more host time per call than the kernel takes on the GPU
        side, fg = torch.cuda.Stream(), torch.cuda.CUDAGraph()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            env.setup_synth(mode, gidf)
            for t in range(48):
                env.step(acts[t])
            torch.cuda.synchronize()
            env.setup_synth(mode, gidf)
            with torch.cuda.graph(fg, stream=side):
                for t in range(48):
                    env.step(acts[t])
        torch.cuda.synchronize()
        for r in range(reps + 2):
            env.setup_synth(mode, gidf)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fg.replay()
            b.record()
            if r >= 2:
                ev.append((a, b))
        env.reset_stats()
        env.score()
        torch.cuda.synchronize()
        same = bool((env.scores[:n] == want_scores).all().item())
        stf = env.stats()
        f_us = max_over_ranks(sum(a.elapsed_time(b) for a, b in ev) / (48 * len(ev))) * 1e3
        livef = int(stf[S_STEPS]) / 48.0
        f_gbs = (BYTES_PER_ENV_STEP + 1) * livef / (f_us * 1e-6) / 1e9
        forced = {"kernel": "k_step<false, POS> (tarok_step: one externally supplied card per live game, legality checked)",
                  "avg_launch_us": f_us, "achieved": f_gbs, "frac": f_gbs / peak, "unit": "GB/s",
                  "algorithmic_bytes_per_env_step": BYTES_PER_ENV_STEP + 1, "scores_equal_random_leg": same,
                  "error_games": int(stf[S_ERRORS]), "traffic": step_traffic(n, mode, "k_step<forced>"),
                  "note": "actions = the cards of a recorded rollout of the same deals, resident on the device ([48, n] uint8); the 48 "
                          "tarok_step calls replayed as one CUDA graph"}
        assert same, "teacher-forced replay of the recorded actions produced different scores"
        del acts, want_scores, fg

    # ---- fused rollout (state in registers; not HBM-bound) -- informational
    fa, fb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    env.rollout(mode, first_game_id=0, fused=True)
    torch.cuda.synchronize()
    fa.record()
    for i in range(5):
        env.rollout(mode, first_game_id=(i + 1) * total + rank * n, fused=True)
    fb.record()
    torch.cuda.synchronize()
    fused_ms = fa.elapsed_time(fb) / 5

    # ---- end to end through the host-buffer C-ABI entries
    env.deal(rank * n)
    perm_h = torch.empty((n, 54), dtype=torch.uint8).pin_memory()
    perm_h.copy_(env.export_perm())
    rng = np.random.default_rng(1234 + rank)
    c_h = torch.from_numpy(rng.integers(1, 4, n, dtype=np.uint8)).pin_memory()
    d_h = torch.from_numpy(rng.integers(0, 4, n, dtype=np.uint8)).pin_memory()
    k_h = torch.from_numpy(rng.integers(0, 4, n, dtype=np.uint8)).pin_memory()
    sc_h = torch.empty((n, 4), dtype=torch.int16).pin_memory()
    st_h = torch.zeros(32, dtype=torch.int64).pin_memory()
    host_cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    pack_threads = max(1, min(64, (os.cpu_count() or host_cores) // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", world)))))
    rec_h, _ = pack_records(perm_h, c_h, d_h, k_h, threads=pack_threads)   # the same deals + contracts as 20-byte records (pinned)

    def e2e_run(kind):
        def once(i):
            gid = i * total + rank * n
            if kind == "records":
                env.rollout_records(rec_h, sc_h, st_h, first_game_id=gid)
            elif kind == "packed":
                env.rollout_host_packed(perm_h, c_h, d_h, k_h, sc_h, st_h, first_game_id=gid, threads=pack_threads)
            else:
                env.rollout_host(perm_h, c_h, d_h, k_h, sc_h, st_h, first_game_id=gid, fused=(kind == "rows"))
            torch.cuda.current_stream().synchronize()                     # the host reads the result
            return int(st_h[S_STEPS])
        for i in range(args.warmup):
            once(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        cnt = 0
        w0 = time.perf_counter()
        e0.record()
        for i in range(args.steps):
            cnt += once(args.warmup + i)
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - w0
        barrier()
        t = max(max_over_ranks(e0.elapsed_time(e1)), max_over_ranks(wall * 1e3) if kind == "packed" else 0.0)
        return sum_over_ranks(cnt) / (t * 1e-3), t / args.steps

    e2e_rows = e2e_run("rows")          # fused kernel behind an 8-chunk upload/compute/download pipeline, 57-byte rows
    e2e_sw = e2e_run("stepwise")        # stepwise kernels, serial upload -> 52 launches -> download
    e2e_rec = e2e_run("records")        # records packed BEFORE the timed region (not end to end for a caller holding rows)
    e2e_packed = e2e_run("packed")      # rows in, packed into records by host threads inside the call, chunk by chunk
    pipes = {"rows": (e2e_rows, world * n * 57), "packed": (e2e_packed, world * n * RECORD_BYTES)}
    best = max(pipes, key=lambda k: pipes[k][0][0])
    clocks = sampler.stop() if sampler else None

    # ---- HBM-bound regime: the same step kernel on a state 8x larger than L2 (informational)
    big = None
    if rank == 0 and not args.no_large:
        try:
            nb = 8 << 20
            eb = TarokEnv(nb, seed=SEED, device=local_rank)
            eb.deal(0); eb.force_contract_synth(mode) if not auction else eb.auction_synth(mode)
            eb.exchange_synth(mode == MODE_AUCTION_UNIFORM)
            eb.step_random(8)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record(); eb.step_random(36); b.record()
            torch.cuda.synchronize()
            us = a.elapsed_time(b) / 36 * 1e3
            live = int(eb.live().sum().item())
            gbs = BYTES_PER_ENV_STEP * live / (us * 1e-6) / 1e9
            tr = step_traffic(nb, mode)
            big = {"games": nb, "state_bytes": nb * 105, "avg_launch_us": us, "achieved": gbs, "frac": gbs / peak, "unit": "GB/s",
                   "traffic": tr, "dram_gbs_from_traffic": (tr / (us * 1e-6) / 1e9) if tr else None,
                   "dram_frac_from_traffic": (tr / (us * 1e-6) / 1e9 / peak) if tr else None}
            eb.close()
        except Exception as ex:    # out of memory on a shared box etc.
            big = {"error": str(ex)[:200]}
    env.close()

    # ---- BASELINE configs 3 and 5 as sub-records: a FIXED total sharded over the ranks by global game id ---------------
    def sharded_leg(total_deals, smode, k_steps):
        first, count = shard(total_deals, rank, world)
        e = TarokEnv(count, seed=SEED, device=local_rank)
        e.set_materialise(False)
        glob = torch.zeros((k_steps + 3, 32), dtype=torch.int64, device=dev)

        def one(i, row):
            e.reset_stats()
            e.setup_synth(smode, i * total_deals + first)
            e.step_random(48)
            e.score()
            comm.allreduce_stats(e, out=glob[row])                          # tarok_allreduce_stats (C ABI, raw NCCL)

        one(0, 0)                                                           # batch 0: global game ids [0, total): the hash
        chk = e.stats_dev.clone()
        if world > 1:
            dist.all_reduce(chk)
        same = bool((chk == glob[0]).all().item())
        g0 = glob[0].cpu().numpy()
        sha = hashlib.sha256(np.ascontiguousarray(g0[:21]).tobytes()).hexdigest()
        one(1, 1); one(2, 2)
        barrier()
        evs = []
        for i in range(k_steps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); one(3 + i, 3 + i); b.record()
            evs.append((a, b))
        barrier()
        t_ms = max_over_ranks(sum(a.elapsed_time(b) for a, b in evs))
        tot = glob[3:3 + k_steps].sum(0).cpu().numpy()
        e.close()
        return {"total_deals": total_deals, "deals_per_gpu": count, "mode": smode, "mode_name": MODE_NAMES.get(smode), "steps": k_steps,
                "ms_per_step": t_ms / k_steps, "env_steps_per_sec": float(tot[S_STEPS]) / (t_ms * 1e-3),
                "deals_per_sec": float(tot[S_FINISHED]) / (t_ms * 1e-3), "scaling": "strong (fixed total, sharded by global game id)",
                "stats_sha256": sha, "batch0_stats": [int(x) for x in g0[:21]],
                "collective": "tarok_allreduce_stats (C ABI, ncclAllReduce int64[32])", "collective_equals_torch_distributed": same}

    sub = {}
    if not args.no_sub:
        ks = max(3, min(args.steps, args.sub_steps))
        try:
            sub["config3"] = {"uniform_bids": sharded_leg(CONFIG3_TOTAL, 17, ks), "bot_bids": sharded_leg(CONFIG3_TOTAL, 18, ks),
                              "workload": "config 3: Berac plus bidding across all Tip_igre contracts, 4,194,304 concurrent deals over the box"}
            sub["config5"] = dict(sharded_leg(CONFIG5_TOTAL, 17, ks),
                                  workload="config 5: full bidding+play, 16,777,216 concurrent deals sharded over the ranks")
        except Exception as ex:
            sub["config3_5_error"] = str(ex)[:300]
        try:
            sub["config4"] = config4_record(local_rank, rank, world, max(2, min(3, args.steps)), dev, max_over_ranks, sum_over_ranks)
        except Exception as ex:
            sub["config4"] = {"error": str(ex)[:300]}
    comm.close()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        r = cpu_port_rate(mode, 12.0)
        cpu = {"value": r["steps_per_s"], "unit": "env-steps/s", "cores": r["cores"], "kind": "port",
               "sample": "%d deals of the same workload (%.1f s, OpenMP over %d threads)" % (r["deals"], r["seconds"], r["cores"]),
               "deals_per_sec": r["deals_per_s"], "single_core_value": r["single_core_steps_per_s"],
               "python_reference_same_box": python_reference_same_box(20.0) if not args.no_pyref else {"status": "skipped (--no-pyref)"}}

    if rank == 0:
        bv, bms = pipes[best][0]
        out = {
            "metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": config_of(args),
            "notes": {
                "outputs": "per-deal scores (int16 x4) + the all-reduced statistics vector = Tarok.rezultati; won-card piles stay "
                           "in the 4-byte-per-trick log (TAROK_OPT_MATERIALISE=0), as Tarok.paralel_start never returns them",
                "l2": ("no flush: every iteration regenerates and revisits its own %d MB state (> 126 MB L2)" % (n * 153 >> 20))
                      if args.no_flush else
                      ("160 MiB flush write between iterations, outside the per-iteration event pairs (and every iteration "
                       "regenerates its own %d MB state, larger than L2); within one iteration the 48 play_steps revisit "
                       "that state as the workload prescribes" % (n * 153 >> 20)),
                "timing": "one step = tarok_rollout_stepwise = one CUDA-graph replay of setup + 48 x play_step + score (TAROK_OPT_GRAPH); "
                          "each of the K steps bracketed by its own CUDA-event pair; ms_per_step = their mean, max over ranks; "
                          "region_ms_incl_flush = first event to last event including the flush writes"},
            "region_ms_incl_flush": region_ms,
            "deals_per_sec": deals / (ms * 1e-3), "env_steps": env_steps, "deals": deals, "error_games": errors,
            "e2e": {"value": bv, "unit": "env-steps/s", "h2d_bytes_per_step": pipes[best][1],
                    "d2h_bytes_per_step": world * (n * 8 + 256), "ms_per_step": bms, "pipeline": best,
                    "api": {"rows": "tarok_rollout_host (TarokEnv.rollout_host): pinned host permutation rows + contracts in, scores + "
                                    "stats out; fused kernel behind an 8-chunk upload/compute/download pipeline",
                            "packed": "tarok_rollout_host_packed: the same rows in; every chunk serialised into 20-byte deal records by "
                                      "%d host threads inside the call, right before its upload" % pack_threads}[best],
                    "rows_57B": {"value": e2e_rows[0], "ms_per_step": e2e_rows[1], "h2d_bytes_per_step": world * n * 57},
                    "rows_packed_in_call_20B": {"value": e2e_packed[0], "ms_per_step": e2e_packed[1], "h2d_bytes_per_step": world * n * RECORD_BYTES,
                                                "pack_threads_per_rank": pack_threads, "host_cores": os.cpu_count(),
                                                "timing": "max(CUDA events, host wall clock) per step: the pack runs on host threads"},
                    "stepwise_kernels": {"value": e2e_sw[0], "ms_per_step": e2e_sw[1]},
                    "records_prepacked": {"value": e2e_rec[0], "ms_per_step": e2e_rec[1], "h2d_bytes_per_step": world * n * RECORD_BYTES,
                                          "note": "tarok_rollout_records with the records packed BEFORE the timed region: an upper bound "
                                                  "for the packed pipeline, NOT an end-to-end number for a caller that holds rows"}},
            "gpu_launches": launches * world,
            "roofline": roofline, "roofline_large": big, "step_forced": forced,
            "fused_rollout": {"ms_per_rollout": fused_ms, "env_steps_per_sec_per_gpu": env_steps / args.steps / world / (fused_ms * 1e-3),
                              "note": "one kernel, state in registers; ALU-bound, no HBM fraction claimed"},
            "abi_collective_ok": abi_collective_ok,
            "cpu_baseline": cpu, "clocks": clocks,
        }
        out.update(sub)
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(out) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


def config4_record(local_rank, rank, world, steps, dev, max_over_ranks, sum_over_ranks):
    """BASELINE config 4 as a sub-record: 65,536 envs per GPU, FOUR players with their own (restated, random-init) nets and
    epsilon; in-scope cost = env kernels + device bucketing + observation expansion + action selection (CUDA events per
    section); the forward passes are the reference's networks (library LSTM/GEMM kernels), reported beside it."""
    import torch
    from tarok_b200.samoigra import Samoigra
    n = CONFIG4_ENVS
    s = Samoigra(n, device=local_rank, seed=SEED, random_card=[0.05, 0.05, 0.05, 0.05], igralci=4)
    s.odigraj(rank * n)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    env_steps, parts, buckets = 0, {}, 0
    for i in range(steps):
        st, ms = s.odigraj((1 + i) * n * world + rank * n, meri=True)
        env_steps += int(st[19])
        buckets += sum(s.zadnji_koraki)
        for k, v in ms.items():
            parts[k] = parts.get(k, 0.0) + v
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    s.zapri()
    per = {k: v / steps for k, v in parts.items()}
    in_scope = per.get("env", 0) + per.get("obs", 0) + per.get("select", 0) + per.get("bucket", 0)
    in_scope = max_over_ranks(in_scope)
    wall = max_over_ranks(wall)
    tot_steps = sum_over_ranks(env_steps)
    return {"workload": "config 4: self-play, four players with their own restated policy nets (random init) forward + GPU env step, "
                        "%d envs per GPU" % n,
            "envs_per_gpu": n, "players": 4, "rollouts": steps, "env_steps_per_rollout_per_gpu": env_steps / steps,
            "device_ms_per_rollout": per, "in_scope_ms_per_rollout": in_scope,
            "obs_plus_select_ms_per_rollout": per.get("obs", 0) + per.get("select", 0) + per.get("bucket", 0),
            "env_steps_per_sec_in_scope": tot_steps / steps / (in_scope * 1e-3),
            "env_steps_per_sec_incl_forwards": tot_steps / wall,
            "forward_buckets_per_rollout": buckets / steps,
            "note": "in scope = env (deal/auction/exchange/step/score kernels) + bucket (device counting sort by (player, net, T), one "
                    "1 KB D2H per step) + obs (observation expansion) + select (action selection); forward = the reference-architecture "
                    "nets (cuDNN LSTM / cuBLAS, out of scope to accelerate)"}


def run_config4(args, local_rank):
    """`--config 4`: only the config-4 record, one JSON line."""
    import torch
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    ident = lambda x: x
    rec = config4_record(local_rank, 0, 1, args.steps, dev, ident, ident)
    print(json.dumps({"metric": "env_steps_per_sec", "value": rec["env_steps_per_sec_incl_forwards"], "unit": "env-steps/s", "n_gpus": 1,
                      "higher_is_better": True, "dtype": "u64 env / fp32 nets", "data": "synthetic", "config4": rec}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100,
                    help="K, the timed steps of the headline rollout loop, of each end-to-end leg and of --config 4; the "
                         "informational legs time min(max(K, 3), 20) forced-action replays, max(3, min(K, --sub-steps)) "
                         "rollouts per config-3/5 sub-record and max(2, min(K, 3)) per config-4 sub-record")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--games", type=int, default=1 << 20, help="concurrent deals per GPU")
    ap.add_argument("--mode", type=int, default=16)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-pyref", action="store_true", help="skip timing the Python reference even where its tree exists")
    ap.add_argument("--no-large", action="store_true")
    ap.add_argument("--no-forced", action="store_true", help="skip the externally-driven k_step<false> leg")
    ap.add_argument("--no-sub", action="store_true", help="skip the config 3 / 4 / 5 sub-records")
    ap.add_argument("--sub-steps", type=int, default=5, help="timed rollouts per sub-record")
    ap.add_argument("--no-flush", action="store_true", help="skip the L2-flush write between iterations (the 159 MB state is larger than L2)")
    ap.add_argument("--config", type=int, default=2, help="2 (default, the headline workload) or 4 (neural self-play only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="config-2 GPU rollout only (not with --impl reference or --config 4): write to DIR as .npy the "
                         "per-deal scores of the last timed step and the statistics vector accumulated over the K timed steps")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.config == 4):
        ap.error("--dump-outputs applies to the GPU rollout of config 2")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.config == 4:
        if rank == 0:
            run_config4(args, local_rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        print("bench.py: --gpus %d needs torchrun (one process per GPU)" % args.gpus, file=sys.stderr)
        sys.exit(2)
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
