#!/usr/bin/env python3
"""bench.py — episodes/s of the batched 2025-2050 rollout + scoring + weight-update step on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--episodes E] [--impl reference]

A step = one training batch: E episodes per GPU (default 65,536 in flight, BASELINE configs[2]) sampled from the
current action-weight table, simulated 2025-2050, scored, and summarised into the update statistics; for N > 1 the
statistics table is summed with one NCCL allreduce (weak scaling: E per GPU). Prints ONE JSON line on rank 0.

  value     episodes/s with everything resident in HBM (kernels + collective only), CUDA-event timed per step,
            L2 flushed between steps, max over ranks
  e2e       episodes/s through BatchTrainer.step(): weights uploaded from the host every step, statistics and the
            batch winner read back, host-side update applied (wall clock between device synchronisations)
  roofline  rollout kernel: algorithmic HBM bytes / measured kernel time vs MEASURED_PEAKS.json (the path is not
            HBM-bound, DESIGN.md §roofline says what binds instead)
  cpu_baseline  the CPU oracle (a port of the reference's Rust loop) on this box's host cores, bounded sample

`--impl reference` times that CPU port alone (rank 0 only) and prints the same line with "impl": "reference".

`--dump-outputs DIR` writes what the last timed step computed on rank 0 as DIR/<name>.npy (float32 / float64, at most 64 MB
in all; larger outputs are a fixed, seeded sample). The inputs depend on the arguments only, so two builds run with the same
arguments can be compared array by array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
ASSETS = os.path.join(ROOT, "tests", "golden", "ireland_map")
METRIC = "full 2025-2050 episodes simulated and scored per second"
UNIT = "episodes/s"
RESULT_BYTES, TRAJ_BYTES, POLICY_BYTES = 64, 1088, 38784
DUMP_SEED = 20250101  # the sample --dump-outputs takes of an output too large to write whole
DUMP_EPISODES, DUMP_RECORDS, DUMP_SITES = 65536, 4096, 4096
DUMP_LIMIT = 64 << 20


def write_outputs(out_dir, arrays):
    """--dump-outputs: every array as out_dir/<name>.npy."""
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT, "outputs of %d bytes exceed the dump limit" % total
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), name
        np.save(os.path.join(out_dir, name + ".npy"), a)


def dump_sample(n, k):
    """Indices of a fixed, seeded sample of k out of n items in ascending order (all of them when n <= k)."""
    import numpy as np
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n, k, replace=False))


def rollout_outputs(results, traj, packs):
    """What a caller of the rollout step receives: every episode's result, the action records, and the exchanged buffer of
    every rank ([update statistics | score, global id and record of the rank's best episode], trainer.PACK_WORDS int64 each).
    The statistics words are counts on the initial weight table, so float64 holds them exactly."""
    import numpy as np
    from eirgrid_b200 import _abi
    out = {}
    pick = dump_sample(len(results), DUMP_EPISODES)
    out["result_episode"] = pick.astype(np.float64)
    for f in ("score", "net_emissions", "public_opinion", "total_cost", "power_reliability", "n_generators", "n_offsets",
              "n_deficit_actions", "n_additional_actions", "flags"):
        out["result_" + f] = results[f][pick].astype(np.float64)
    pick = dump_sample(len(traj), DUMP_RECORDS)
    out["traj_episode"] = pick.astype(np.float64)
    for f in ("n_deficit", "n_additional", "actions"):
        out["traj_" + f] = traj[f][pick].astype(np.float32)
    out["update_stats"] = packs[:, :_abi.STATS_WORDS].sum(axis=0).astype(np.float64)
    out["rank_best_score"] = packs[:, _abi.STATS_WORDS].copy().view(np.float64)
    out["rank_best_episode"] = packs[:, _abi.STATS_WORDS + 1].astype(np.float64)
    return out


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons while the timed regions run."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.stop = threading.Event()
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.02)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(timeout=3)

    def summary(self):
        sm = sorted(float(r[1]) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def cpu_reference_rate(seconds_target, threads, literal=True, mode_fast=False):
    """episodes/s of the CPU oracle (port of the reference loop) on a bounded sample."""
    import oracle_lib as O
    w = O.World.ireland(fast=True)
    ow = O.Weights()
    mode = O.FAST if mode_fast else O.FAITHFUL
    n = max(threads * 2, 8)
    t0 = time.perf_counter()
    w.rollout(ow, n, seed=20250101, mode=mode, literal_scan=literal and not mode_fast, threads=threads, want_sites=False, want_yearly=False)
    dt = time.perf_counter() - t0
    rate = n / dt
    n2 = int(max(n, min(rate * seconds_target, 4_000_000)))
    t0 = time.perf_counter()
    w.rollout(ow, n2, seed=20250101, first_episode=n, mode=mode, literal_scan=literal and not mode_fast, threads=threads, want_sites=False,
              want_yearly=False)
    dt = time.perf_counter() - t0
    return n2 / dt, n2, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    import oracle_lib as O
    threads = os.cpu_count() or 1
    w = O.World.ireland(fast=True)
    ow = O.Weights()
    # size one step so that the whole run (warm-up + K steps) is about a minute of CPU work, at most 2 s per step
    probe = max(threads, 4)
    t0 = time.perf_counter()
    w.rollout(ow, probe, seed=20250101, mode=O.FAITHFUL, literal_scan=True, threads=threads, want_sites=False, want_yearly=False)
    step_seconds = min(2.0, 60.0 / max(args.steps + args.warmup, 1))
    per_step = max(probe, int(probe / (time.perf_counter() - t0) * step_seconds))
    per_step = max(2 * threads, (per_step + threads - 1) // threads * threads)  # whole rounds of the thread pool
    first = probe
    for _ in range(args.warmup):
        w.rollout(ow, per_step, seed=20250101, first_episode=first, mode=O.FAITHFUL, literal_scan=True, threads=threads, want_sites=False, want_yearly=False)
        first += per_step
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res, traj, _, _ = w.rollout(ow, per_step, seed=20250101, first_episode=first, mode=O.FAITHFUL, literal_scan=True, threads=threads,
                                    want_sites=False, want_yearly=False)
        ow.update(res, traj)  # the write-lock section, sequential like the reference
        first += per_step
    dt = time.perf_counter() - t0
    value = args.steps * per_step / dt
    sample = "%d steps x %d episodes, literal 100x100 placement scan + sequential weight update, %d threads" % (args.steps, per_step, threads)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "policy rollout + scoring + batch weight-update statistics, %d episodes in flight per GPU "
                                   "(BASELINE configs[2] batch shape), Irish map: 130 settlements, 59 existing plants, 2601 candidate sites" % args.episodes,
                       "map": "ireland", "episodes_per_step": per_step,
                       "reference_arm": "CPU oracle port of the reference loop (the Rust reference cannot be built here): literal 100x100 placement "
                                        "scan, per-evaluation opinion sums, sequential per-episode weight update; each step is a bounded sample of the workload"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


SUIT_METRIC = "candidate generator sites analysed per second (15 types x 26 years each)"
SUIT_UNIT = "sites/s"


def suitability_workload_text(args, info):
    return ("location suitability of every candidate generator site: %d x %d sites over the 50 km map (%.1f m apart) x 15 generator types x 26 "
            "simulated years, %s map (%d settlements, %d existing plants, %d coastline points), sites sharded over the ranks"
            % (args.sites_per_axis, args.sites_per_axis, 50000.0 / max(args.sites_per_axis - 1, 1), args.suitability_map,
               info["n_settlements"], info["n_existing"], info["n_coast"]))


def cpu_suitability_rate(seconds_target):
    """sites/s (26 years each) of the CPU oracle's calculate_generator_suitability port on a bounded sample: the oracle
    analyses analyze_map's 51 x 51 grid of one year per pass, as the reference does; the points of a pass are split over all
    host threads (the oracle call releases the GIL)."""
    from concurrent.futures import ThreadPoolExecutor
    import oracle_lib as O
    w = O.World.ireland(fast=False)
    threads = os.cpu_count() or 1
    n_points = 2601
    cuts = [n_points * t // threads for t in range(threads + 1)]

    def one_pass(pool):
        list(pool.map(lambda t: w.location_analysis(1, first=cuts[t], n=cuts[t + 1] - cuts[t]), range(threads)))

    with ThreadPoolExecutor(threads) as pool:
        t0 = time.perf_counter()
        one_pass(pool)
        one = time.perf_counter() - t0
        passes = int(max(1, min(seconds_target / max(one, 1e-9), 5000)))
        t0 = time.perf_counter()
        for _ in range(passes):
            one_pass(pool)
        dt = time.perf_counter() - t0
    site_years = passes * n_points
    return site_years / 26.0 / dt, "%d passes x 2601 points x 1 year in %.1f s (= %d site-years), %d threads" % (passes, dt, site_years, threads), threads, dt


def run_reference_suitability(args):
    if int(os.environ.get("RANK", 0)) != 0:
        return
    rate, sample, threads, dt = cpu_suitability_rate(min(2.0 * max(args.steps, 1), 60.0))
    line = {"impl": "reference", "metric": SUIT_METRIC, "value": rate, "unit": SUIT_UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / max(args.steps, 1) * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": "location suitability of every candidate generator site x 15 types x 26 years (BASELINE configs[4])",
                       "reference_arm": "CPU oracle port of Map::calculate_generator_suitability (the Rust reference cannot be built here), one "
                                        "analyze_map pass per simulated year like the reference; bounded sample"},
            "cpu_baseline": {"value": rate, "unit": SUIT_UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": rate, "unit": SUIT_UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def run_suitability(args, emit):
    """BASELINE configs[4]: all candidate sites x 15 types x 26 years, sharded by site over the ranks, one final all-gather."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from eirgrid_b200 import _lib, synthetic, trainer as T

    world = int(os.environ.get("WORLD_SIZE", 1))
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    stream = torch.cuda.Stream(dev)
    ctx = _lib.Context(local, stream.cuda_stream)
    if args.suitability_map == "scaled10":
        ctx.map_set(*synthetic.scaled_map(ASSETS, factor=10))
    else:
        ctx.map_load_dir(ASSETS)
    info = ctx.map_info()
    side = args.sites_per_axis
    step = 50000.0 / max(side - 1, 1)
    n_sites = side * side
    NY, NT = 26, 15
    first, n_mine = T.shard_of(n_sites, rank, world)
    per_site = NY * NT  # doubles
    # equal-sized slots for the gather: the largest shard
    slot = T.shard_of(n_sites, 0, world)[1]
    d_mine = torch.zeros(slot * per_site, dtype=torch.float64, device=dev)
    d_all = torch.zeros(world * slot * per_site, dtype=torch.float64, device=dev) if world > 1 else d_mine
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def one_pass():
        ctx.location_analysis_sites(True, side, step, 0, NY, first, n_mine, d_scores=d_mine)
        if world > 1:
            with torch.cuda.stream(stream):
                dist.all_gather_into_tensor(d_all, d_mine)

    W, K = max(args.warmup, 3), args.steps
    for _ in range(W):
        one_pass()
    barrier()
    with ClockSampler(local) as clocks:
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(K)]
        launches0 = ctx.kernel_launches()
        barrier()
        for k in range(K):
            with torch.cuda.stream(stream):
                flush.zero_()
            ev[k][0].record(stream)
            ctx.location_analysis_sites(True, side, step, 0, NY, first, n_mine, d_scores=d_mine)
            ev[k][1].record(stream)
            if world > 1:
                with torch.cuda.stream(stream):
                    dist.all_gather_into_tensor(d_all, d_mine)
            ev[k][2].record(stream)
        barrier()
        launches = ctx.kernel_launches() - launches0
        if args.dump_outputs and rank == 0:  # this rank's scores of a seeded sample of its sites
            pick = dump_sample(n_mine, DUMP_SITES)
            outputs = {"site": (first + pick).astype(np.float64),
                       "scores": d_mine.view(-1, NY, NT)[torch.from_numpy(pick).to(dev)].cpu().numpy()}
        t = torch.tensor([sum(ev[k][0].elapsed_time(ev[k][2]) for k in range(K)), sum(ev[k][0].elapsed_time(ev[k][1]) for k in range(K))],
                         dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        step_ms, kernel_ms = float(t[0].item()) / K, float(t[1].item()) / K
        value = n_sites / (step_ms / 1e3)
        # e2e: the host-buffer entry point (scores copied to the host inside the call), this rank's shard
        Ke = min(K, 3)
        barrier()
        t0 = time.perf_counter()
        for _ in range(Ke):
            host_scores = ctx.location_analysis_sites(True, side, step, 0, NY, first, n_mine)
        barrier()
        e2e_s = time.perf_counter() - t0
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e = n_sites * Ke / float(t.item())
        # the placement search's own candidate grid (51 x 51 sites at 1 km), all 26 years: a single small launch
        small = torch.zeros(2601 * per_site, dtype=torch.float64, device=dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctx.location_analysis_sites(True, 51, 1000.0, 0, NY, 0, 2601, d_scores=small)
        barrier()
        e0.record(stream)
        for _ in range(20):
            ctx.location_analysis_sites(True, 51, 1000.0, 0, NY, 0, 2601, d_scores=small)
        e1.record(stream)
        barrier()
        small_ms = e0.elapsed_time(e1) / 20
    clock_summary = clocks.summary()
    # a checksum of the gathered scores: every rank must hold the same table
    import hashlib
    torch.cuda.synchronize()
    if world > 1:
        # ranks' slots are `slot` sites long; drop the padding of the shorter shards
        parts = [d_all[r * slot * per_site:(r * slot + T.shard_of(n_sites, r, world)[1]) * per_site] for r in range(world)]
        full = torch.cat(parts)
    else:
        full = d_mine[:n_sites * per_site]
    sha = hashlib.sha256(full.cpu().numpy().tobytes()).hexdigest()[:16]
    water_sites = int((full.view(-1, NY, NT)[:, 0, 1] > 0).sum().item())  # OffshoreWind scores > 0 exactly on water tiles
    if world > 1:
        shas = [None] * world
        dist.all_gather_object(shas, sha)
        assert len(set(shas)) == 1, "ranks hold different score tables: %s" % shas
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak, peak_src = load_peaks()
    n_coast = info["n_coast"]
    # algorithmic work of one launch: every site tests 1 + 9 + 9 probes against every polygon edge, a site on water 441 more
    # (get_distance_to_nearest_land); the scores are written once, 15 x 26 doubles per site (DESIGN.md)
    mine_frac = n_mine / n_sites
    edge_tests = n_coast * (19 * n_sites + 441 * water_sites) * mine_frac
    algo_bytes = n_mine * per_site * 8 + (2 * n_coast + 2 * info["n_settlements"]) * 8 + 26 * info["n_settlements"] * 12
    achieved = algo_bytes / (kernel_ms / 1e3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "suitability_traffic.json")
    if os.path.exists(tp):
        prof = json.load(open(tp))
        if prof.get("sites_per_launch") == n_sites and world == prof.get("n_gpus", 1) and args.suitability_map == "ireland":
            traffic = prof.get("dram_bytes_per_launch")
    line = {"metric": SUIT_METRIC, "value": value, "unit": SUIT_UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": step_ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": suitability_workload_text(args, info), "sites": n_sites, "sites_on_water": water_sites,
                       "scores_per_step": n_sites * per_site, "kernel_ms": kernel_ms, "gather_ms": step_ms - kernel_ms,
                       "l2": "256 MiB buffer written between timed steps (L2 flush)",
                       "timing": "CUDA events on the launching stream per step, max over ranks",
                       "placement_grid_51x51_all_years_ms": small_ms, "scores_sha256_16": sha},
            "e2e": {"value": e2e, "unit": SUIT_UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": n_mine * per_site * 8,
                    "what": "eg_location_analysis_sites with a HOST output buffer: kernel + device-to-host copy of this rank's scores inside the call"},
            "gpu_launches": int(launches), "clocks": clock_summary,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "peak_source": peak_src, "kernel": "eg_suitability_kernel (+ eg_suit_rows_kernel, the crossing lists)", "algorithmic_bytes_per_launch": algo_bytes,
                         "edge_tests": {"per_launch": edge_tests, "g_per_s": edge_tests / (kernel_ms / 1e3) / 1e9,
                                        "what": "ALGORITHMIC point-in-polygon edge tests (const_funcs.rs:143-158): 19 probes per site + 441 per site on "
                                                "water, each against every coastline edge, as the reference performs them; the kernel answers a probe by "
                                                "binary search in the sorted crossing list of its row instead (same result, ~7 comparisons)"},
                         "note": "the scores written (3.1 KB per site) are the only HBM traffic that scales; after the crossing-list restructuring the "
                                 "kernel's time is the per-site settlement / plant distance loops, the reductions over years and the score stores "
                                 "(profiles/r02_suitability.md)"}}
    if world == 1 and not args.no_cpu_baseline:
        rate, sample, threads, _ = cpu_suitability_rate(args.cpu_seconds)
        line["cpu_baseline"] = {"value": rate, "unit": SUIT_UNIT, "cores": threads, "kind": "port", "sample": sample}
    if args.dump_outputs:
        write_outputs(args.dump_outputs, outputs)
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--episodes", type=int, default=65536, help="episodes in flight per GPU per step")
    ap.add_argument("--impl", default="eirgrid_b200")
    ap.add_argument("--seed", type=int, default=20250101)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", choices=["ireland", "scaled10", "suitability"], default="ireland",
                    help="ireland: shipped map, 65,536 episodes in flight per GPU (BASELINE configs[2] batch shape, the headline); "
                         "scaled10: synthetic 10x scaled grid of configs[3] (eirgrid_b200/synthetic.py); "
                         "suitability: configs[4], every candidate site x 15 types x 26 years, sharded by site over the ranks")
    ap.add_argument("--total-episodes", type=int, default=0,
                    help="fixed-total mode (configs[3]: 1,000,000): every step is this many episodes split over the ranks (strong scaling)")
    ap.add_argument("--sites-per-axis", type=int, default=1001,
                    help="suitability workload: candidate sites per axis over the 50 km map (51 = the placement search's own 1 km grid)")
    ap.add_argument("--suitability-map", choices=["ireland", "scaled10"], default="ireland")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed on rank 0 as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU implementation")
    if args.impl == "reference":
        return run_reference_suitability(args) if args.workload == "suitability" else run_reference(args)

    # stdout carries exactly one JSON line: libraries that print to fd 1 (NCCL's version banner) go to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        os.write(json_fd, (json.dumps(line) + "\n").encode())

    if args.workload == "suitability":
        return run_suitability(args, emit)

    import torch
    import torch.distributed as dist
    from eirgrid_b200 import trainer as T

    world = int(os.environ.get("WORLD_SIZE", 1))
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    map_arrays = None
    if args.workload == "scaled10":
        from eirgrid_b200 import synthetic
        map_arrays = synthetic.scaled_map(ASSETS, factor=10)
    strong = args.total_episodes > 0
    if strong:  # fixed total per step, split over the ranks (the first total % world ranks take one episode more)
        args.episodes = T.shard_of(args.total_episodes, 0, world)[1]
    tr = T.BatchTrainer(args.episodes, seed=args.seed, device=local, asset_dir=ASSETS, map_arrays=map_arrays, distributed=world > 1)
    n_total = args.total_episodes if strong else args.episodes * world
    tr.set_batch(n_total)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=tr.device)  # > 126 MB L2

    def first_of(step_index):  # global id of this rank's first episode in batch `step_index` (batches never share ids)
        return step_index * n_total + tr.offset

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    W = max(args.warmup, 3)
    K = args.steps
    tr.upload_weights()  # value is measured on the initial action-weight table (first batch of a training run)
    for k in range(W):
        tr.launch_rollout(first_episode=first_of(k))
        tr.launch_stats()
        tr.reduce_stats()
        tr.warm_exchange()  # first-use costs of the small torch ops / collectives of step(), weights untouched
    barrier()

    with ClockSampler(local) as clocks:
        # ---- value: device-resident step (rollout + statistics kernels [+ allreduce]), CUDA events per step -------
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(K)]
        launches0 = tr.ctx.kernel_launches()
        barrier()
        for k in range(K):
            with torch.cuda.stream(tr.stream):
                flush.zero_()
            ev[k][0].record(tr.stream)
            tr.launch_rollout(first_episode=first_of(W + k))
            ev[k][1].record(tr.stream)
            tr.launch_stats()
            ev[k][3].record(tr.stream)
            tr.exchange()  # the one exchange of the step: [statistics | best-episode record] of every rank onto every rank
            ev[k][2].record(tr.stream)
        barrier()
        launches = tr.ctx.kernel_launches() - launches0
        tr.check_exchange()
        if args.dump_outputs and rank == 0:  # the later sections reuse the trainer's buffers: copy the last step out now
            res_last, traj_last = tr.fetch_results()
            outputs = rollout_outputs(res_last, traj_last, tr.d_all_pack.cpu().numpy().reshape(world, T.PACK_WORDS))
        step_ms = sum(ev[k][0].elapsed_time(ev[k][2]) for k in range(K))
        rollout_ms = sum(ev[k][0].elapsed_time(ev[k][1]) for k in range(K)) / K
        collective_us = sum(ev[k][3].elapsed_time(ev[k][2]) for k in range(K)) / K * 1e3
        t = torch.tensor([step_ms], dtype=torch.float64, device=tr.device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        step_ms = float(t.item())
        value = n_total * K / (step_ms / 1e3)

        # ---- e2e: the public training step, host weights in, statistics out, host update applied ----------------
        barrier()
        t0 = time.perf_counter()
        for _ in range(K):
            tr.step()
        barrier()
        e2e_s = time.perf_counter() - t0
        t = torch.tensor([e2e_s], dtype=torch.float64, device=tr.device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
        e2e = n_total * K / e2e_s
        # every rank applied the same update to its own copy of the weights: the tables must be identical, bit for bit
        import hashlib
        weights_sha = hashlib.sha256(bytes(tr.weights.table())).hexdigest()[:16]
        if world > 1:
            shas = [None] * world
            dist.all_gather_object(shas, weights_sha)
            assert len(set(shas)) == 1, "ranks ended the e2e steps with different weight tables: %s" % shas

        # ---- e2e with every episode's result and action record copied to the host (SimulationResult per episode)
        res_h = torch.empty(args.episodes * RESULT_BYTES, dtype=torch.uint8).pin_memory()
        traj_h = torch.empty(args.episodes * TRAJ_BYTES, dtype=torch.uint8).pin_memory()
        barrier()
        t0 = time.perf_counter()
        for _ in range(K):
            tr.upload_weights()
            tr.launch_rollout()
            with torch.cuda.stream(tr.stream):
                res_h.copy_(tr.d_results, non_blocking=True)
                traj_h.copy_(tr.d_traj, non_blocking=True)
            tr.stream.synchronize()
        barrier()
        full_s = time.perf_counter() - t0

        # ---- the general kernel: every year's YearlyMetrics computed and written (eg_yearly, 3.7 KB per episode) -----------
        KY = min(K, 10)
        d_yearly = torch.empty(tr.n * 3744, dtype=torch.uint8, device=tr.device)
        evy = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(KY)]
        tr.ctx.rollout_device(tr.n, tr.seed, first_of(5000), tr.d_results, tr.d_traj, None, d_yearly, tr.cfg)
        barrier()
        for k in range(KY):
            with torch.cuda.stream(tr.stream):
                flush.zero_()
            evy[k][0].record(tr.stream)
            tr.ctx.rollout_device(tr.n, tr.seed, first_of(5001 + k), tr.d_results, tr.d_traj, None, d_yearly, tr.cfg)
            evy[k][1].record(tr.stream)
        barrier()
        t = torch.tensor([sum(evy[k][0].elapsed_time(evy[k][1]) for k in range(KY))], dtype=torch.float64, device=tr.device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        value_yearly = n_total * KY / (float(t.item()) / 1e3)
        del d_yearly

        # ---- the reference's own update rule: one snapshot, the batch rolled out, every record applied in episode order on
        # the GPU (eg_train_batch_inorder). Sequential in the episodes, so several ranks would only replicate: rank-local.
        inorder = None
        if world == 1:
            KI = min(K, 10)
            w_keep = tr.weights
            tr.weights = T._lib.Weights()
            tr.step_inorder(tr.n, rng_seed=args.seed)
            barrier()
            t0 = time.perf_counter()
            for _ in range(KI):
                tr.step_inorder(tr.n, rng_seed=args.seed)
            barrier()
            dt = time.perf_counter() - t0
            inorder = {"value": tr.n * KI / dt, "unit": UNIT, "ms_per_step": dt / KI * 1e3,
                       "what": "eg_train_batch_inorder: snapshot H2D, rollout, the reference's per-episode update (learning.rs:131-373) applied "
                               "in episode order by the GPU, state D2H; bit-identical to the host rule (tests/test_gpu_update_inorder.py)"}
            tr.weights = w_keep

        # ---- the device-resident step again on the table the e2e steps have trained (what explains e2e vs value) ---------
        KT = min(K, 20)
        tr.upload_weights()
        evt = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(KT)]
        barrier()
        for k in range(KT):
            with torch.cuda.stream(tr.stream):
                flush.zero_()
            evt[k][0].record(tr.stream)
            tr.launch_rollout(first_episode=first_of(W + K + k + 1000))
            tr.launch_stats()
            tr.reduce_stats()
            evt[k][1].record(tr.stream)
        barrier()
        t = torch.tensor([sum(evt[k][0].elapsed_time(evt[k][1]) for k in range(KT))], dtype=torch.float64, device=tr.device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        value_trained = n_total * KT / (float(t.item()) / 1e3)
    clock_summary = clocks.summary()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = load_peaks()
    info = tr.ctx.map_info()
    ns = info["grid_n"] ** 2
    # algorithmic HBM bytes of one rollout launch (DESIGN.md §4.1): every episode writes its result and action record
    # once; the static tables (walk lists 16 B + order 2 B per (class, year, site), per-site factors, plant terms, small
    # tables, stamp pattern, policy snapshot) are read once and then live in L2
    static_bytes = 7 * 26 * ns * (16 + 2) + ns * 16 + 26 * 15 * 3 * 26 * 16 + 40000 + 3200 + POLICY_BYTES
    algo_bytes = tr.n * (RESULT_BYTES + TRAJ_BYTES) + static_bytes
    achieved = algo_bytes / (rollout_ms / 1e3) / 1e9
    traffic, issue = None, None
    tp = os.path.join(ROOT, "profiles", "rollout_traffic.json")
    if os.path.exists(tp):
        try:
            prof = json.load(open(tp))
            if args.workload != "ireland":
                raise KeyError("profile is for the shipped map")
            if prof.get("episodes_per_launch") == args.episodes:
                traffic = prof.get("dram_bytes_per_launch")
            # what binds instead of HBM: warp-instruction issue. Instructions per episode are a property of the code and
            # the workload (counted by ncu, profiles/), the rate is measured live here.
            sms, sched = torch.cuda.get_device_properties(local).multi_processor_count, 4
            ipe = prof["warp_instructions_per_episode"]
            peak_issue = sms * sched * (clock_summary.get("sm_mhz") or 1965.0) * 1e6
            issue = {"warp_instructions_per_episode": ipe, "achieved_ginst_s": ipe * tr.n / (rollout_ms / 1e3) / 1e9,
                     "peak_ginst_s": peak_issue / 1e9, "frac": ipe * tr.n / (rollout_ms / 1e3) / peak_issue,
                     "source": "profiles/rollout_traffic.json (ncu smsp__inst_executed.sum) x live kernel time"}
            # FP64 ceiling without FMA (the path is compiled --fmad=false), measured live; the kernel's share of it from ncu
            import ctypes
            peak64 = ctypes.c_double()
            if T._lib.lib().eg_microbench_fp64(local, ctypes.byref(peak64)) == 0:
                issue["fp64_peak_tflops_no_fma"] = peak64.value
                issue["fp64_pipe_active_pct"] = prof.get("fp64_pipe_pct")
            # the second resource the kernel runs close to (ncu, same capture): the L1 / shared-memory data pipe
            issue["l1_data_pipe_busy_pct_ncu"] = prof.get("l1_data_pipe_pct")
            issue["issue_slots_busy_pct_ncu"] = prof.get("issue_active_pct")
            issue["resident_warps_per_sm_ncu"] = prof.get("resident_warps_per_sm")
        except Exception:
            traffic, issue = None, None
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": step_ms / K, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": "policy rollout + scoring + batch weight-update statistics, %d episodes in flight per GPU "
                               "(BASELINE configs[2] batch shape), %s" % (args.episodes, "Irish map: 130 settlements, 59 existing plants, 2601 candidate sites"
                                                                          if args.workload == "ireland" else
                                                                          "synthetic 10x scaled grid (configs[3]): %d settlements, %d existing plants, %d candidate sites"
                                                                          % (info["n_settlements"], info["n_existing"], ns)),
                   "map": args.workload,
                   "episodes_per_gpu": args.episodes, "l2": "256 MiB buffer written between timed steps (L2 flush)",
                   "timing": "CUDA events on the launching stream per step, max over ranks",
                   "rollout_kernel_ms": rollout_ms,
                   "value_on_trained_table": value_trained,
                   "value_with_yearly_metrics": value_yearly,
                   "collective": {"what": "one exchange of [statistics int64[5156] | best-episode record 1168 B] per step onto every rank, summed locally in rank order",
                                  "how": tr.exchange_kind,
                                  "bytes_per_rank": tr.pack_words * 8, "us_per_step": collective_us if world > 1 else 0.0},
                   "weights_sha256_16_after_e2e": weights_sha,
                   "episodes_per_step_total": n_total},
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": POLICY_BYTES, "d2h_bytes_per_step": tr.d2h_bytes_per_step,
                "what": "BatchTrainer.step(): weights H2D from the host, rollout + statistics + winner-record kernels, statistics and "
                        "winner record D2H (pinned), host-side weight update applied. The weights learn during these steps (stagnation-mode "
                        "tables sample ~20 % more actions and plants per episode), so the rollout itself is slower here than in `value`, "
                        "which is timed on the initial table",
                "with_all_results_to_host": {"value": n_total * K / full_s, "unit": UNIT,
                                             "d2h_bytes_per_step": args.episodes * (RESULT_BYTES + TRAJ_BYTES)},
                "reference_rule_in_order_on_gpu": inorder},
        "gpu_launches": int(launches),
        "clocks": clock_summary,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "peak_source": peak_src, "kernel": "eg_episode_kernel<REPLAY=false, GEOM, MODE=1> (rollout, lean training instantiation)",
                     "algorithmic_bytes_per_launch": algo_bytes, "issue": issue,
                     "note": "the path moves ~1.2 KB per episode and is bound by warp-instruction issue/latency, not HBM: "
                             "see roofline.issue, DESIGN.md §4.1 and profiles/"},
    }
    if strong:
        line["config"]["workload"] += "; fixed total of %d episodes per step split over the ranks" % n_total
    if world == 1 and not args.no_cpu_baseline and args.workload == "ireland":
        threads = os.cpu_count() or 1
        rate, n_cpu, dt = cpu_reference_rate(args.cpu_seconds, threads, literal=True)
        rate_fast, n_fast, dt_fast = cpu_reference_rate(3.0, threads, mode_fast=True)
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": "%d episodes in %.1f s, oracle in reference-cost mode (literal 100x100 placement scan, per-evaluation opinion sums), %d threads"
                                          % (n_cpu, dt, threads),
                                "fast_mode": {"value": rate_fast, "sample": "%d episodes in %.1f s with the exact table restructurings" % (n_fast, dt_fast)}}
    if args.dump_outputs:
        write_outputs(args.dump_outputs, outputs)
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
