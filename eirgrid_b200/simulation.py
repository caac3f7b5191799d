"""Host driver mirroring the reference's run_multi_simulation (core/multi_simulation.rs:95-1242) for the hot path.

Same arguments and on-disk layout as the reference's batch loop:
  <checkpoint_dir>/<2024%m%d_%H%M%S>/{latest_weights.json, checkpoint_iteration.txt, best_weights.json,
                                       weight_history.json (with --track-weight-history)}
and the same resume rule (newest directory whose name is 15 characters of digits/'_' with year <= 2025,
multi_simulation.rs:210-290,385-413). The rayon `into_par_iter` over iterations becomes batches of episodes on
the GPU(s); CSV export, console reports and the interactive full-simulation prompt are out of scope
(SURVEY.md §8(f) N2).
"""
import datetime
import glob
import json
import os
import time

import numpy as np

from . import _abi, _lib

FULL_RUN_PERCENTAGE = 10                  # multi_simulation.rs:38
REPLAY_BEST_STRATEGY_IN_FULL_RUNS = True  # multi_simulation.rs:39


def run_dir_name(now=None):
    """Timestamp directory name: literal "2024" + %m%d_%H%M%S (multi_simulation.rs:161-163)."""
    now = now or datetime.datetime.now()
    return "2024" + now.strftime("%m%d_%H%M%S")


def _valid_run_dir(name):
    # multi_simulation.rs:219-234
    if len(name) != 15 or not all(c.isdigit() or c == "_" for c in name):
        return False
    try:
        year, month, day = int(name[0:4]), int(name[4:6]), int(name[6:8])
    except ValueError:
        return False
    return not (year > 2025 or month > 12 or day > 31)


def find_resume_dir(checkpoint_dir):
    """Newest checkpoint directory the reference would resume from, or None."""
    if not os.path.isdir(checkpoint_dir):
        return None
    names = [n for n in os.listdir(checkpoint_dir) if os.path.isdir(os.path.join(checkpoint_dir, n)) and _valid_run_dir(n)]
    return os.path.join(checkpoint_dir, max(names)) if names else None


def find_start_iteration(checkpoint_dir):
    """multi_simulation.rs:385-413: checkpoint_iteration.txt of the max directory whose name is digits/'_' only."""
    if not os.path.isdir(checkpoint_dir):
        return 0
    names = [n for n in os.listdir(checkpoint_dir)
             if os.path.isdir(os.path.join(checkpoint_dir, n)) and all(c.isdigit() or c == "_" for c in n)]
    if not names:
        return 0
    path = os.path.join(checkpoint_dir, max(names), "checkpoint_iteration.txt")
    if not os.path.exists(path):
        return 0
    try:
        return int(open(path).read().strip())
    except ValueError:
        return 0


_LOOK = object()


def load_initial_weights(checkpoint_dir, continue_from_checkpoint=True, log=print, resume_dir=_LOOK):
    """latest_weights.json overlaid with every thread_*_weights.json (multi_simulation.rs:237-290).
    resume_dir: the directory to resume from when the caller has already chosen it (None = none found)."""
    if not continue_from_checkpoint:
        log("Starting fresh simulation (--no-continue specified)")
        return _lib.Weights()
    latest = find_resume_dir(checkpoint_dir) if resume_dir is _LOOK else resume_dir
    if latest is None:
        log("No checkpoint directories found, starting fresh")
        return _lib.Weights()
    merged, found = _lib.Weights(), False
    shared = os.path.join(latest, "latest_weights.json")
    if os.path.exists(shared):
        try:
            merged, found = _lib.Weights.load_from_file(shared), True
        except _lib.EirgridError:
            pass
    for path in sorted(glob.glob(os.path.join(latest, "thread_*_weights.json"))):
        try:
            merged.update_weights_from(_lib.Weights.load_from_file(path))
            found = True
        except _lib.EirgridError:
            pass
    if not found:
        log("No weights found in latest directory, starting fresh")
        return _lib.Weights()
    return merged


def _best_score(weights):
    t = weights.table()
    if not t.has_best:
        return None
    import math
    net, opinion, cost = t.best_metrics[0], t.best_metrics[1], t.best_metrics[2]
    if net > 0.0:
        return 1.0 - min(net / 1000000.0, 1.0)
    normalized = max(cost / 50000000000.0, 1.0)
    cs = 1.0 - min(math.log(normalized) / math.log(100.0), 1.0)
    cw = 0.8 if normalized > 8.0 else 0.5
    return 1.0 + (cs * cw + opinion * (1.0 - cw))


def run_multi_simulation(asset_dir, num_iterations, parallel=True, continue_from_checkpoint=True,
                         checkpoint_dir="checkpoints", checkpoint_interval=5, progress_interval=10, cache_dir="cache",
                         force_full_simulation=False, seed=None, verbose_logging=False, optimization_mode=None,
                         enable_energy_sales=True, enable_csv_export=True, debug_weights=False,
                         enable_construction_delays=False, track_weight_history=False,
                         batch_size=65536, update_mode="batch", master_seed=None, device=None, log=print):
    """Run `num_iterations` episodes (total across all ranks) and learn the action weights.

    update_mode "batch": device-side statistics + one allreduce per batch (DESIGN.md §update).
    update_mode "sequential": the reference's per-episode update in episode order, applied on the GPU (eg_update_device:
    exact reference rule with `batch_size` episodes sampled per snapshot; replicated on every rank).
    The replay phase (last 10 % of the iterations) always runs the per-episode rule.
    Returns a summary dict; checkpoints are written like the reference's.
    """
    import torch
    import torch.distributed as dist
    from .trainer import BatchTrainer

    distributed = dist.is_available() and dist.is_initialized()
    rank = dist.get_rank() if distributed else 0
    world = dist.get_world_size() if distributed else 1
    if update_mode not in ("batch", "sequential"):
        raise ValueError("update_mode must be 'batch' or 'sequential'")
    os.makedirs(checkpoint_dir, exist_ok=True)
    # Everything a run derives from the clock or from the checkpoint directory is decided by rank 0 and broadcast: ranks that
    # looked for themselves could pick different seeds, or see rank 0's new (empty) run directory as the one to resume from.
    same_stream = seed is not None  # quirk Q8: --seed re-seeds every episode with the same value
    if rank == 0:
        plan = {"resume_dir": find_resume_dir(checkpoint_dir) if continue_from_checkpoint else None,
                "start_iteration": find_start_iteration(checkpoint_dir) if continue_from_checkpoint else 0,
                "run_dir": os.path.join(checkpoint_dir, run_dir_name()),
                "cache_loaded": os.path.exists(os.path.join(cache_dir, "location_analysis.json")),  # load_location_analysis, :149-154
                "rng_seed": int(seed) if seed is not None else int(master_seed if master_seed is not None else time.time_ns() & 0xFFFFFFFFFFFF)}
    else:
        plan = None
    if distributed and world > 1:
        box = [plan]
        dist.broadcast_object_list(box, src=0)
        plan = box[0]
    weights = load_initial_weights(checkpoint_dir, continue_from_checkpoint, log if rank == 0 else (lambda *a: None),
                                   resume_dir=plan["resume_dir"])
    if distributed and world > 1:
        dist.barrier()  # every rank has read the old checkpoint before rank 0 creates the new directory next to it
    start_iteration, run_dir, cache_loaded, rng_seed = plan["start_iteration"], plan["run_dir"], plan["cache_loaded"], plan["rng_seed"]
    if rank == 0:
        os.makedirs(run_dir, exist_ok=True)
        if track_weight_history and not os.path.exists(os.path.join(run_dir, "weight_history.json")):
            open(os.path.join(run_dir, "weight_history.json"), "w").write("[]")
    if rank == 0 and not cache_loaded:
        log("Warning: Location analysis cache not found in %s. All simulations will use full mode." % cache_dir)
    per_gpu = max(1, min(int(batch_size), (max(num_iterations - start_iteration, 1) + world - 1) // world))
    trainer = BatchTrainer(per_gpu, seed=rng_seed, device=device, weights=weights, asset_dir=asset_dir,
                           distributed=distributed)
    trainer.next_episode = start_iteration
    final_full = (num_iterations * FULL_RUN_PERCENTAGE) // 100
    completed = start_iteration
    t_start, t_progress = time.time(), time.time()
    next_checkpoint = (completed // checkpoint_interval + 1) * checkpoint_interval
    history = []
    n_flagged = 0
    if rank == 0:
        log("Starting multi-simulation optimization with %d iterations (%d completed, %d remaining) in directory %s"
            % (num_iterations, start_iteration, num_iterations - start_iteration, run_dir))
    while completed < num_iterations:
        is_full_run = force_full_simulation or not cache_loaded or completed >= max(num_iterations - final_full, 0)
        replay_best = is_full_run and REPLAY_BEST_STRATEGY_IN_FULL_RUNS and weights.has_best_actions()
        trainer.cfg = _abi.RunCfg(cost_only=optimization_mode == "cost_only", enable_energy_sales=enable_energy_sales,
                                  enable_construction_delays=enable_construction_delays, replay_best=replay_best,
                                  same_stream_all_episodes=same_stream)
        # never past the requested iteration count, nor past the start of the replay phase: the last batch is smaller, and
        # ragged over the ranks (the first `remainder` ranks take one episode more)
        phase_end = num_iterations if (is_full_run or final_full >= num_iterations) else num_iterations - final_full
        if update_mode == "batch" and not replay_best:
            advance = min(per_gpu * world, phase_end - completed)
            trainer.set_batch(advance)
            st = trainer.step()
        else:
            # Replay batches and the sequential mode run the reference's per-episode rule (it rebuilds the doubled records of
            # replay iterations, quirk Q10). The rule is sequential in the episodes: with several ranks the ROLLOUT of the batch is
            # sharded and the records are all-gathered, then every rank applies the same in-order update to the whole batch on
            # its own GPU (identical inputs, identical tables, no further exchange).
            advance = min(per_gpu * world, phase_end - completed)
            st = trainer.step_inorder_sharded(advance, rng_seed=rng_seed)
        completed += advance
        n_flagged += int(st.n_flagged)
        if st.n_flagged and rank == 0:
            log("warning: %d episodes of this batch carry eg_result.flags (replay-phase years with more than 40 recorded actions, "
                "quirk Q10; or a capacity overflow)" % st.n_flagged)
        if rank == 0:
            if time.time() - t_progress >= progress_interval:
                t_progress = time.time()
                rate = (completed - start_iteration) / max(time.time() - t_start, 1e-9)
                log("Progress: %d/%d iterations, %.0f iterations/s, best score %s" % (completed, num_iterations, rate, _best_score(weights)))
            if completed >= next_checkpoint or completed >= num_iterations:
                next_checkpoint = (completed // checkpoint_interval + 1) * checkpoint_interval
                weights.save_to_file(os.path.join(run_dir, "latest_weights.json"))
                open(os.path.join(run_dir, "checkpoint_iteration.txt"), "w").write(str(min(completed, num_iterations)))
                if track_weight_history:
                    weights.history_append(completed, os.path.join(run_dir, "weight_history.json"))
    elapsed = time.time() - t_start
    csv_dir = None
    if rank == 0:
        weights.save_to_file(os.path.join(run_dir, "best_weights.json"))  # multi_simulation.rs:1161-1163
        if enable_csv_export and weights.has_best_actions():  # multi_simulation.rs:852-925
            csv_dir = trainer.ctx.export_best_run_csv(weights, os.path.join(run_dir, "enhanced_csv"),
                                                      _abi.RunCfg(cost_only=optimization_mode == "cost_only", enable_energy_sales=enable_energy_sales))
    t = weights.table()
    summary = {"run_dir": run_dir, "iterations": completed, "start_iteration": start_iteration, "elapsed_s": elapsed,
               "episodes_per_s": (completed - start_iteration) / max(elapsed, 1e-9), "best_score": _best_score(weights),
               "best_metrics": {"final_net_emissions": t.best_metrics[0], "average_public_opinion": t.best_metrics[1],
                                "total_cost": t.best_metrics[2], "power_reliability": t.best_metrics[3]} if t.has_best else None,
               "iterations_without_improvement": t.iterations_without_improvement, "n_gpus": world, "csv_dir": csv_dir, "flagged_episodes": n_flagged}
    trainer.close()
    return summary
