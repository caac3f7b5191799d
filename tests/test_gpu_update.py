"""GPU tests of the batch-synchronous update: statistics kernel vs its numpy restatement, BatchTrainer steps."""
import os

import numpy as np
import pytest

import oracle_lib as O
import stats_ref
from eirgrid_b200 import _abi, _lib

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ASSETS = os.path.join(ROOT, "tests", "golden", "ireland_map")


def _best_lists(w):
    has, b, d = w.best()
    return [x.tolist() for x in b], [x.tolist() for x in d]


@pytest.mark.parametrize("iwi", [0, 40, 900])
def test_stats_kernel_matches_numpy(gpu_ctx, oracle_world, iwi):
    import torch
    n = 300
    gw = _lib.Weights()
    res0, traj0, _, _ = oracle_world.rollout(O.Weights(), 32, seed=41)
    gw.update(res0, traj0)
    t = gw.table()
    t.iterations_without_improvement = iwi
    gw.set_table(t)
    res, traj, _, _ = gpu_ctx.rollout(gw, n, seed=42)
    dev = torch.device("cuda", 0)
    d_res = torch.from_numpy(res.view(np.uint8).copy()).to(dev)
    d_traj = torch.from_numpy(traj.view(np.uint8).copy()).to(dev)
    d_stats = torch.zeros(_abi.STATS_WORDS, dtype=torch.int64, device=dev)
    d_bs = torch.zeros(1, dtype=torch.float64, device=dev)
    d_bi = torch.zeros(1, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    gpu_ctx.weights_upload(gw)
    gpu_ctx.update_stats_device(gw, n, d_res, d_traj, d_stats, d_bs, d_bi)
    gpu_ctx.sync()
    got = d_stats.cpu().numpy()
    consts = stats_ref.contrast_consts(t)
    best, best_def = _best_lists(gw)
    exp, scores, terms = stats_ref.batch_stats(res, traj, consts, best, best_def)
    assert got[0] == n
    stats_ref.assert_stats_match(got, float(d_bs.item()), int(d_bi.item()) % (1 << 64), exp, scores, terms)


def test_trainer_steps_learn_and_are_deterministic():
    from eirgrid_b200 import trainer as T
    tr = T.BatchTrainer(4096, seed=7, device=0, asset_dir=ASSETS)
    s1 = tr.step()
    assert s1.n_episodes == 4096 and s1.n_improvements == 1 and s1.best_score > 1.0
    t1 = bytes(tr.weights.table())
    res, traj = tr.fetch_results()
    assert (res["flags"] == 0).all() and (res["power_reliability"] == 1.0).all()
    # the stored best strategy is the batch winner's record
    k = s1.batch_best_episode
    has, b, d = tr.weights.best()
    for y, (dd, aa) in enumerate(_abi.traj_rows(traj[k])):
        assert b[y].tolist() == dd.tolist() + aa.tolist() and d[y].tolist() == dd.tolist()
    s2 = tr.step()
    assert tr.weights.table().iteration_count == 8192
    assert s2.best_score >= s1.best_score
    w = tr.weights.table().arrays()[0]
    assert w.min() >= 0.0001 and w.max() <= 0.999
    tr.close()
    tr2 = T.BatchTrainer(4096, seed=7, device=0, asset_dir=ASSETS)
    tr2.step()
    assert bytes(tr2.weights.table()) == t1
    tr2.close()


def test_batch_rule_score_distribution_matches_sequential_rule(gpu_ctx):
    """North star (2): final scores of the batch-synchronous rule agree with the reference's sequential rule across seeds.
    Measured gap at 8k-65k iterations: 0.001-0.002 with sigma 0.0015-0.0025 (profiles/r01_learning_distribution.md)."""
    from eirgrid_b200 import trainer as T
    n_iter, seeds = 4096, (2001, 2002, 2003, 2004)

    def best(w):
        t = w.table()
        assert t.has_best and t.best_metrics[0] <= 0.0 and t.best_metrics[3] == 1.0  # net-zero and reliable
        return stats_ref.default_score(*list(t.best_metrics)[:3])

    seq, bat = [], []
    for s in seeds:
        w = _lib.Weights()
        for first in range(0, n_iter, 16):  # 16 stale workers, per-episode update in order
            res, traj, _, _ = gpu_ctx.rollout(w, 16, seed=s, first_episode=first)
            w.update(res, traj, rng_seed=s)
        seq.append(best(w))
        tr = T.BatchTrainer(256, seed=s, device=0, asset_dir=ASSETS)
        for _ in range(n_iter // 256):
            tr.step()
        bat.append(best(tr.weights))
        tr.close()
    assert abs(np.mean(seq) - np.mean(bat)) < 0.01, (seq, bat)
    assert min(bat) > 1.88 and min(seq) > 1.88


def test_flagged_episodes_are_counted(gpu_ctx):
    """Episodes that exceed a fixed capacity (or find no site) are counted in the update statistics of both update paths."""
    import torch
    rs = np.random.RandomState(5)
    n = 64
    t = np.zeros(n, _abi.TRAJ_DTYPE)
    t["n_additional"][:8, :] = 37
    t["actions"][:8, :26 * 37] = rs.randint(0, 45, (8, 26 * 37))   # 962 plants: over the 560-plant capacity
    t["n_additional"][8:, 0] = 1
    res, _, _ = gpu_ctx.replay(t)
    assert int((res["flags"] != 0).sum()) == 8
    w = _lib.Weights()
    assert w.update(res, t).n_flagged == 8              # sequential path
    dev = torch.device("cuda", 0)
    d_res = torch.from_numpy(res.view(np.uint8).copy()).to(dev)
    d_traj = torch.from_numpy(t.view(np.uint8).copy()).to(dev)
    d_stats = torch.zeros(_abi.STATS_WORDS, dtype=torch.int64, device=dev)
    d_bs = torch.zeros(1, dtype=torch.float64, device=dev)
    d_bi = torch.zeros(1, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    w2 = _lib.Weights()
    gpu_ctx.weights_upload(w2)
    gpu_ctx.update_stats_device(w2, n, d_res, d_traj, d_stats, d_bs, d_bi)
    gpu_ctx.sync()
    stats = d_stats.cpu().numpy()
    assert stats[0] == n and stats[2] == 8               # batch path: header word 2
