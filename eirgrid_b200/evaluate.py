"""Policy evaluation: how good is a policy table? Score, per-year outcome and action statistics of a checkpoint over many episodes,
rolled out and reduced on the GPU (eg_evaluate), without copying episodes to the host.

    python -m eirgrid_b200.evaluate --weights best_weights.json --assets tests/golden/ireland_map -n 1048576 --json eval.json
    torchrun --nproc-per-node 8 -m eirgrid_b200.evaluate --weights best_weights.json --assets ... -n 100000000

Under torch.distributed every rank evaluates its contiguous share of the episode ids (trainer.shard_of), the ranks all-gather
their records and every rank merges them in rank order (eg_eval_stats_merge), so all ranks hold the same bytes.
"""
import argparse
import os
import sys
import tempfile

import numpy as np

from . import _abi, _lib
from .trainer import shard_of


def evaluate_policy(weights, n, ctx, seed=1, first_episode=0, cfg=None, with_yearly=True, dist=None):
    """EvalStats of episodes first_episode .. first_episode + n - 1. `dist`: an initialised torch.distributed (or None for one
    process); the ranks share the ids and end with the same merged record."""
    world = dist.get_world_size() if dist else 1
    rank = dist.get_rank() if dist else 0
    offset, count = shard_of(n, rank, world)
    mine = ctx.evaluate(weights, count, seed=seed, first_episode=first_episode + offset, cfg=cfg, with_yearly=with_yearly)
    if world == 1:
        return mine
    import torch
    size = _abi.C.sizeof(_abi.EvalStats)
    dev = torch.device("cuda", torch.cuda.current_device())
    local = torch.from_numpy(np.frombuffer(bytes(mine), np.uint8).copy()).to(dev)
    gathered = torch.empty(world * size, dtype=torch.uint8, device=dev)
    dist.all_gather_into_tensor(gathered, local)
    raw = gathered.cpu().numpy()
    out = _abi.EvalStats()
    for r in range(world):
        out.merge(_abi.EvalStats.from_bytes(raw[r * size:(r + 1) * size]))
    return out


def _unsigned(text):
    if not text.isdigit():
        raise argparse.ArgumentTypeError("invalid value '%s': expected an unsigned integer" % text)
    return int(text)


def parse_args(argv=None):
    ap = argparse.ArgumentParser(prog="python -m eirgrid_b200.evaluate",
                                 description="Statistics of a policy table over many episodes, reduced on the GPU")
    ap.add_argument("--weights", required=True, help="policy table (ActionWeights JSON, e.g. best_weights.json)")
    ap.add_argument("--assets", required=True, help="directory with settlements.json, ireland_generators.csv, coastline_points.json")
    ap.add_argument("-n", "--episodes", type=_unsigned, required=True)
    ap.add_argument("--seed", type=_unsigned, default=1)
    ap.add_argument("--first-episode", type=_unsigned, default=0)
    ap.add_argument("--cost-only", action="store_true", default=False, help="score with optimization_mode cost_only")
    ap.add_argument("--no-yearly", action="store_true", default=False, help="skip the per-year statistics (faster)")
    ap.add_argument("--json", default=None, help="write the statistics here (default: print them)")
    return ap.parse_args(argv)


def main(argv=None):
    args = parse_args(argv)
    world = int(os.environ.get("WORLD_SIZE", 1))
    rank = int(os.environ.get("RANK", 0))
    dist = None
    device = 0
    try:
        if world > 1:
            import torch
            import torch.distributed as dist
            device = int(os.environ.get("LOCAL_RANK", 0))
            torch.cuda.set_device(device)
            dist.init_process_group("nccl", device_id=torch.device("cuda", device))
        ctx = _lib.Context(device)
        ctx.map_load_dir(args.assets)
        weights = _lib.Weights.load_from_file(args.weights)
        st = evaluate_policy(weights, args.episodes, ctx, seed=args.seed, first_episode=args.first_episode,
                             cfg=_abi.RunCfg(cost_only=args.cost_only), with_yearly=not args.no_yearly, dist=dist)
        if rank == 0:
            if args.json:
                st.write_json(args.json)
            else:
                with tempfile.TemporaryDirectory() as tmp:
                    path = os.path.join(tmp, "evaluation.json")
                    st.write_json(path)
                    sys.stdout.write(open(path).read())
        ctx.close()
    except _lib.EirgridError as e:
        print("error: %s" % e, file=sys.stderr)
        return 1
    finally:
        if dist is not None:
            dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
