"""Time of a policy evaluation (eg_evaluate) against a rollout of the same episodes with the same outputs requested
(eg_rollout_batch_device), and the reduction kernels' own time, on one GPU. Prints one JSON line and writes it to --out.

    python scripts/eval_time.py --out profiles/r03_eval_time.json [-n 1048576] [--reps 5]

Rollout: one eg_rollout_batch_device call of n episodes into device buffers (results + action records, plus the per-year records
for the yearly mode), timed with the host clock around the call and a stream synchronisation. Evaluation: eg_evaluate of the
same ids (snapshot upload, chunked rollout + reduction, one copy of the record to the host), timed the same way. Reduction:
eg_eval_accumulate_device over the rollout's device outputs, timed with CUDA events on the context's stream. Every
configuration is warmed up once; repetitions alternate between the configurations and the median is reported. The card's
name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from eirgrid_b200 import _abi, _lib  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("-n", type=int, default=1 << 20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("eval_time.py needs a CUDA device (no CPU fallback)")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(dev)
    ctx = _lib.Context(0, stream.cuda_stream)
    ctx.map_load_dir(os.path.join(ROOT, "tests", "golden", "ireland_map"))
    w = _lib.Weights()
    n = args.n
    u8 = torch.uint8
    d_res = torch.empty(n * _abi.RESULT_DTYPE.itemsize, dtype=u8, device=dev)
    d_traj = torch.empty(n * _abi.TRAJ_DTYPE.itemsize, dtype=u8, device=dev)
    d_yearly = torch.empty(n * _abi.YEARLY_DTYPE.itemsize, dtype=u8, device=dev)
    d_acc = torch.zeros(_abi.C.sizeof(_abi.EvalStats), dtype=u8, device=dev)
    torch.cuda.synchronize(dev)

    def rollout(yearly):
        ctx.weights_upload(w)
        ctx.sync()
        t0 = time.perf_counter()
        ctx.rollout_device(n, args.seed, 0, d_res, d_traj, None, d_yearly if yearly else None)
        ctx.sync()
        return time.perf_counter() - t0

    def evaluate(yearly):
        t0 = time.perf_counter()
        ctx.evaluate(w, n, seed=args.seed, with_yearly=yearly)
        return time.perf_counter() - t0

    def reduction(yearly):  # over the outputs of the last rollout(yearly)
        with torch.cuda.stream(stream):
            d_acc.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
        ctx.eval_accumulate_device(n, d_res, d_traj, d_yearly if yearly else None, 0, d_acc)
        with torch.cuda.stream(stream):
            e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / 1e3

    times = {k: [] for k in ("rollout_traj", "evaluate_traj", "reduce_traj", "rollout_yearly", "evaluate_yearly", "reduce_yearly")}
    for rep in range(args.reps + 1):  # repetition 0 is the warm-up
        for yearly, tag in ((False, "traj"), (True, "yearly")):
            r = rollout(yearly)
            k = reduction(yearly)
            e = evaluate(yearly)
            if rep:
                times["rollout_" + tag].append(r)
                times["reduce_" + tag].append(k)
                times["evaluate_" + tag].append(e)
    med = {k: float(np.median(v)) for k, v in times.items()}
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    line = {
        "what": "policy evaluation vs rollout of the same episodes, one GPU",
        "episodes": n, "reps": args.reps, "device": torch.cuda.get_device_name(0),
        "nvidia_smi_name_power_limit": smi.stdout.strip() or None,
        "median_s": med,
        "episodes_per_s": {k: n / v for k, v in med.items() if not k.startswith("reduce")},
        "evaluate_over_rollout_rate": {tag: med["rollout_" + tag] / med["evaluate_" + tag] for tag in ("traj", "yearly")},
        "reduction_share_of_rollout": {tag: med["reduce_" + tag] / med["rollout_" + tag] for tag in ("traj", "yearly")},
        "all_s": times,
    }
    text = json.dumps(line)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
