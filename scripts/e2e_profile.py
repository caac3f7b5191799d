#!/usr/bin/env python3
"""Per-phase timing of BatchTrainer.step() over a few batches (weights evolve as in training)."""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from eirgrid_b200 import trainer as T  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 6
tr = T.BatchTrainer(n, seed=20250101, device=0, asset_dir=os.path.join(ROOT, "tests", "golden", "ireland_map"))
for s in range(steps):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    t0 = time.perf_counter()
    tr.upload_weights()
    t1 = time.perf_counter()
    ev[0].record(tr.stream)
    tr.launch_rollout()
    ev[1].record(tr.stream)
    tr.launch_stats()
    ev[2].record(tr.stream)
    tr.exchange()
    with torch.cuda.stream(tr.stream):
        tr.h_all_pack.copy_(tr.d_all_pack, non_blocking=True)
    ev[3].record(tr.stream)
    tr.stream.synchronize()
    t2 = time.perf_counter()
    st = T.sum_and_apply(tr.weights, tr.h_all_pack.numpy(), n, tr.next_episode)
    tr.next_episode += n
    t3 = time.perf_counter()
    res, traj = tr.fetch_results()
    print("step %d: upload %.2f ms | rollout %.2f ms | stats %.2f ms | exchange+d2h %.2f ms | host apply %.2f ms | total %.2f ms | "
          "iwi %d best %.4f improved %d | mean gens %.1f actions/ep %.1f flags %d" % (
              s, (t1 - t0) * 1e3, ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3]), (t3 - t2) * 1e3,
              (t3 - t0) * 1e3, st.iterations_without_improvement, st.best_score, st.n_improvements,
              res["n_generators"].mean(), (res["n_deficit_actions"].astype(float) + res["n_additional_actions"]).mean(), int((res["flags"] != 0).sum())))
