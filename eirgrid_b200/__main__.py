"""Command line of the aiSimulator hot path: same flag names and defaults as the reference's clap struct
(aiSimulator/src/cli/cli.rs:3-59), plus --assets / --batch-size / --update-mode / --master-seed.

    python -m eirgrid_b200 -n 100000 --assets tests/golden/ireland_map --no-continue
    torchrun --nproc-per-node 8 -m eirgrid_b200 -n 1000000 ...
"""
import argparse
import json
import os
import sys


def _unsigned(text):
    # clap's usize/u64: decimal digits only
    if not text.isdigit():
        raise argparse.ArgumentTypeError("invalid value '%s': expected an unsigned integer" % text)
    return int(text)


def _positive(text):
    v = _unsigned(text)
    if v == 0:
        raise argparse.ArgumentTypeError("must be positive")
    return v


def parse_args(argv=None):
    ap = argparse.ArgumentParser(prog="eirgrid_b200", description="EirGrid Power System Simulator (2025-2050), B200 episode engine")
    ap.add_argument("-n", "--iterations", type=_unsigned, default=1000)
    ap.add_argument("-p", "--parallel", action="store_true", default=True)
    ap.add_argument("--no-continue", action="store_true", default=False)
    ap.add_argument("-c", "--checkpoint-dir", default="checkpoints")
    ap.add_argument("-i", "--checkpoint-interval", type=_positive, default=5)
    ap.add_argument("-r", "--progress-interval", type=_unsigned, default=10)
    ap.add_argument("-C", "--cache-dir", default="cache")
    ap.add_argument("--force-full-simulation", action="store_true", default=False)
    ap.add_argument("--enable-timing", action="store_true", default=False)
    ap.add_argument("--seed", type=_unsigned, default=None, help="Random seed for deterministic simulation")
    ap.add_argument("-v", "--verbose-state-logging", action="store_true", default=False)
    ap.add_argument("--cost-only", action="store_true", default=False, help="Optimize for cost only, ignoring emissions and public opinion")
    ap.add_argument("--enable-energy-sales", action="store_true", default=True, help="Enable revenue from energy sales to offset costs")
    ap.add_argument("--enable-csv-export", action="store_true", default=True, help="Enable CSV export of detailed simulation results")
    ap.add_argument("--debug-logging", action="store_true", default=False)
    ap.add_argument("--debug-weights", action="store_true", default=False)
    ap.add_argument("--enable-construction-delays", action="store_true", default=False)
    ap.add_argument("--track-weight-history", action="store_true", default=False)
    # additions of this implementation
    ap.add_argument("--assets", default=os.path.join("aiSimulator", "assets"), help="directory with settlements.json, ireland_generators.csv, coastline_points.json")
    ap.add_argument("--batch-size", type=_positive, default=65536, help="episodes in flight per GPU")
    ap.add_argument("--update-mode", choices=["batch", "sequential"], default="batch")
    ap.add_argument("--master-seed", type=_unsigned, default=None, help="seed of the per-episode RNG streams when --seed is not given")
    return ap.parse_args(argv)


def main(argv=None):
    args = parse_args(argv)
    import torch
    import torch.distributed as dist
    from .simulation import run_multi_simulation
    world = int(os.environ.get("WORLD_SIZE", 1))
    if world > 1:
        local = int(os.environ.get("LOCAL_RANK", 0))
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    print("EirGrid Power System Simulator (2025-2050)")
    summary = run_multi_simulation(
        args.assets, args.iterations, args.parallel, not args.no_continue, args.checkpoint_dir, args.checkpoint_interval,
        args.progress_interval, args.cache_dir, args.force_full_simulation, args.seed, args.verbose_state_logging,
        "cost_only" if args.cost_only else None, args.enable_energy_sales, args.enable_csv_export, args.debug_weights,
        args.enable_construction_delays, args.track_weight_history, batch_size=args.batch_size,
        update_mode=args.update_mode, master_seed=args.master_seed)
    if int(os.environ.get("RANK", 0)) == 0:
        print(json.dumps(summary, indent=2))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
