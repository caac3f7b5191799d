"""The batch kernels of a training step against plain references, at the benchmark's size and on inputs no rollout produces.

- eg_stats_kernel / eg_stats_argbest_kernel (csrc/stats.cu) against tests/stats_ref.py: 65,536 episodes (several trips of
  the grid-stride loop per warp), every score regime, the cost-only mode, best lists longer than the record (quirk Q10),
  records whose counts run past the capacity, ties for the best score, empty and odd-sized batches, accumulation.
- eg_stats_pack_best_kernel byte for byte against trainer.pack_record.
- Which instantiation of eg_episode_kernel the launcher picks, read from a CUDA profiler trace.

The statistics kernel reads only (results, records) from device memory and the uploaded policy, so most inputs are built by
hand. The best lists come from the uploaded policy and the constants from the weights passed with the call: both are the
same weights here.
"""
import json
import re

import numpy as np
import pytest

import oracle_lib as O
import stats_ref
from eirgrid_b200 import _abi, _lib, synthetic
from eirgrid_b200 import trainer as T

pytestmark = pytest.mark.gpu
SCALE_N = 65536
FIRST_GLOBAL = 5 * (1 << 32) + 7  # a global episode id whose two 32-bit halves are both non-zero


def _torch():
    import torch
    return torch


def _dev(a):
    torch = _torch()
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).to(torch.device("cuda", 0))


def _best_lists(w):
    _, b, d = w.best()
    return [x.tolist() for x in b], [x.tolist() for x in d]


def _with_iwi(w, iwi):
    w = w.clone()
    t = w.table()
    t.iterations_without_improvement = iwi
    w.set_table(t)
    return w


class _Stats:
    """One call of the statistics kernel on device copies of (results, records); n may be smaller than the buffers."""

    def __init__(self, ctx, w, res, traj, n=None, d_stats=None):
        torch = _torch()
        dev = torch.device("cuda", 0)
        self.n = len(res) if n is None else n
        self.d_res, self.d_traj = _dev(res), _dev(traj)
        self.d_stats = torch.zeros(_abi.STATS_WORDS, dtype=torch.int64, device=dev) if d_stats is None else d_stats
        self.d_bs = torch.zeros(1, dtype=torch.float64, device=dev)
        self.d_bi = torch.zeros(1, dtype=torch.int64, device=dev)
        torch.cuda.synchronize()
        ctx.weights_upload(w)
        ctx.update_stats_device(w, self.n, self.d_res, self.d_traj, self.d_stats, self.d_bs, self.d_bi)
        ctx.sync()
        self.stats = self.d_stats.cpu().numpy()
        self.best_score = float(self.d_bs.item())
        self.best_index = int(self.d_bi.item()) % (1 << 64)


def _check(ctx, w, res, traj, cost_only=False):
    got = _Stats(ctx, w, res, traj)
    exp, scores, terms = stats_ref.batch_stats(res, traj, stats_ref.contrast_consts(w.table(), cost_only), *_best_lists(w))
    stats_ref.assert_stats_match(got.stats, got.best_score, got.best_index, exp, scores, terms)
    return got, exp, scores


@pytest.fixture(scope="module")
def trained(oracle_world):
    """Weights with a best strategy (one oracle batch and one update)."""
    w = _lib.Weights()
    res, traj, _, _ = oracle_world.rollout(O.Weights(), 32, seed=41)
    w.update(res, traj)
    assert w.table().has_best
    return w


def _make_best(res, i):
    """The highest score there is: net zero, cost within budget, full public support (2.0)."""
    res["net_emissions"][i], res["total_cost"][i], res["public_opinion"][i] = -1.0, 4.0e10, 1.0


@pytest.fixture(scope="module")
def scale_batch(gpu_ctx, trained):
    """65,536 episodes rolled out from the trained table, with results rewritten so that every score regime occurs."""
    res, traj, _, _ = gpu_ctx.rollout(trained, SCALE_N, seed=42)
    e = np.arange(SCALE_N)
    hi = e % 5 == 1  # net <= 0, cost above 8 x 5e10: cost weight 0.8
    res["net_emissions"][hi] = -1000.0
    res["total_cost"][hi] = 4.1e11 + e[hi] * 1e8  # up to 7e12: the log term also reaches its clamp at 1
    pos = e % 5 == 2  # net > 0
    res["net_emissions"][pos] = 1.0 + (e[pos] % 997) * 1000.0
    lo = e % 5 == 3  # net <= 0, cost below 5e10: the cost term is exactly 1
    res["net_emissions"][lo] = -1.0
    res["total_cost"][lo] = 4.0e10
    res["public_opinion"][lo] = np.minimum(res["public_opinion"][lo], 0.999)
    # the one best episode sits on a late trip of the grid-stride loop (148 SMs x 4 blocks x 8 warps = 4,736 warps)
    _make_best(res, 60001)
    return res, traj


def test_stats_at_benchmark_scale(gpu_ctx, trained, scale_batch):
    """65,536 episodes, iwi = 900: every episode passes the contrast test (force), episodes better than the best strategy
    collapse both log words to -2^40 (quirk Q9), the others add their penalties."""
    res, traj = scale_batch
    w = _with_iwi(trained, 900)
    got, exp, scores = _check(gpu_ctx, w, res, traj)
    best = stats_ref.contrast_consts(w.table())["best_score"]
    assert (scores > best).any() and (scores < best).any()
    assert (res["net_emissions"] > 0).any() and (res["total_cost"] > 4e11).any() and (res["total_cost"] < 5e10).any()
    assert got.best_index == 60001 and exp[1] == SCALE_N


def test_stats_cost_only_mode(gpu_ctx, trained, scale_batch, tmp_path):
    """Weights whose checkpoint says "optimization_mode": "cost_only" score episodes and the best strategy by cost alone."""
    path = str(tmp_path / "w.json")
    _with_iwi(trained, 40).save_to_file(path)
    d = json.load(open(path))
    d["optimization_mode"] = "cost_only"
    json.dump(d, open(path, "w"))
    w = _lib.Weights.load_from_file(path)
    res, traj = scale_batch
    _, exp, scores = _check(gpu_ctx, w, res[:8192], traj[:8192], cost_only=True)
    assert 0 < exp[1] < 8192 and scores.max() == 2.0


def test_stats_best_lists_longer_than_the_record(gpu_ctx, oracle_world, trained, scale_batch):
    """The winner of a replay-best batch, adopted with replay_best=True, stores every action twice (quirk Q10): its lists are
    longer than a record's run, and positions past the run are compared with the stored best lists."""
    rb, tb, _, _ = gpu_ctx.rollout(trained, 64, seed=77, cfg=_abi.RunCfg(replay_best=1))
    w = _lib.Weights()
    w.update(rb, tb, replay_best=True)
    w = _with_iwi(w, 900)
    b, d = _best_lists(w)
    res, traj = scale_batch
    rows = [stats_ref.recorded_rows(t) for t in traj[:4096]]
    assert any(len(b[y]) > len(r[y][0]) + len(r[y][1]) for r in rows for y in range(26))
    _check(gpu_ctx, w, res[:4096], traj[:4096])


def test_stats_records_past_the_capacity(gpu_ctx, trained, scale_batch):
    """Counts that run past the 984 slots of a record are cut where the host update cuts them, in a year's deficit part or
    its additional part."""
    rs = np.random.RandomState(9)
    n = 96
    t = np.zeros(n, _abi.TRAJ_DTYPE)
    t["n_deficit"] = rs.randint(0, 50, (n, 26))
    t["n_additional"] = rs.randint(0, 50, (n, 26))
    t["actions"] = rs.randint(0, _abi.N_ACTIONS, (n, _abi.TRAJ_CAPACITY))
    t["n_deficit"][0, 0] = 2000           # cut inside the first year's deficit part
    t["n_deficit"][1], t["n_additional"][1] = 0, 0
    t["n_additional"][1, :24] = 41        # exactly 984 slots
    used = t["n_deficit"].sum(axis=1) + t["n_additional"].sum(axis=1)
    assert (used > _abi.TRAJ_CAPACITY).sum() > n // 2
    res = scale_batch[0][:n].copy()
    for iwi in (40, 900):
        _check(gpu_ctx, _with_iwi(trained, iwi), res, t)


def test_stats_ties_take_the_lowest_index(gpu_ctx, trained, scale_batch):
    """4,737 episodes (one more than the warps of a 148-SM grid) with the best score at three indices, and a batch of
    identical episodes (same_stream_all_episodes = 1)."""
    n = 4737
    res, traj = scale_batch[0][:n].copy(), scale_batch[1][:n]
    for i in (4736, 1000, 33):
        _make_best(res, i)
    got, _, _ = _check(gpu_ctx, _with_iwi(trained, 40), res, traj)
    assert got.best_index == 33
    same_r, same_t, _, _ = gpu_ctx.rollout(trained, 1024, seed=5, cfg=_abi.RunCfg(same_stream_all_episodes=1))
    assert (same_r.view(np.uint8).reshape(len(same_r), -1) == same_r[:1].view(np.uint8)).all()
    got, _, _ = _check(gpu_ctx, _with_iwi(trained, 900), same_r, same_t)
    assert got.best_index == 0


def test_stats_edges_and_accumulation(gpu_ctx, trained, scale_batch):
    torch = _torch()
    res, traj = scale_batch
    w = _with_iwi(trained, 40)
    # one episode
    _check(gpu_ctx, w, res[7:8], traj[7:8])
    # n = 0 (one-element buffers): the table is left as it was, the best score and index are reset
    first = _Stats(gpu_ctx, w, res[:300], traj[:300])
    before = first.stats.copy()
    empty = _Stats(gpu_ctx, w, res[:1], traj[:1], n=0, d_stats=first.d_stats)
    assert np.array_equal(empty.stats, before)
    assert empty.best_score == -1.0 and empty.best_index == (1 << 64) - 1
    # a second call without a clear adds to the table; a clear zeroes it
    second = _Stats(gpu_ctx, w, res[300:1000], traj[300:1000], d_stats=first.d_stats)
    alone = _Stats(gpu_ctx, w, res[300:1000], traj[300:1000])
    assert np.array_equal(second.stats, before + alone.stats)
    gpu_ctx.update_stats_clear_device(first.d_stats)
    gpu_ctx.sync()
    assert not first.d_stats.cpu().numpy().any()
    torch.cuda.synchronize()


def test_pack_best_record(gpu_ctx, trained, scale_batch):
    """The winner record is [best score | first global id + best index | result | record] of the stats kernel's winner; an
    empty shard packs score -1.0, which the combine step never picks over a shard with episodes."""
    torch = _torch()
    res, traj = scale_batch
    w = _with_iwi(trained, 900)
    s = _Stats(gpu_ctx, w, res, traj)
    d_rec = torch.zeros(T.REC_BYTES, dtype=torch.uint8, device=torch.device("cuda", 0))
    gpu_ctx.update_pack_best_device(s.n, s.d_res, s.d_traj, s.d_bs, s.d_bi, FIRST_GLOBAL, d_rec)
    gpu_ctx.sync()
    k = s.best_index
    rec = d_rec.cpu().numpy()
    assert rec.tobytes() == T.pack_record(s.best_score, FIRST_GLOBAL + k, res[k:k + 1], traj[k:k + 1]).tobytes()
    # a shard of no episodes: the kernel reads element 0 of its one-element buffers
    e = _Stats(gpu_ctx, w, res[:1], traj[:1], n=0)
    d_empty = torch.zeros(T.REC_BYTES, dtype=torch.uint8, device=torch.device("cuda", 0))
    gpu_ctx.update_pack_best_device(0, e.d_res, e.d_traj, e.d_bs, e.d_bi, FIRST_GLOBAL, d_empty)
    gpu_ctx.sync()
    empty = d_empty.cpu().numpy()
    assert empty[:8].view(np.float64)[0] == -1.0 and empty[8:16].view(np.int64)[0] == FIRST_GLOBAL
    for recs in ((empty, rec), (rec, empty)):
        st = T.combine_and_apply(w.clone(), s.stats, np.stack(recs), SCALE_N, FIRST_GLOBAL)
        assert st.batch_best_episode == k
    # the record is written in 64-bit words: a buffer that is not 8-byte aligned is refused without a launch
    launches = gpu_ctx.kernel_launches()
    with pytest.raises(_lib.EirgridError) as e:
        gpu_ctx.update_pack_best_device(s.n, s.d_res, s.d_traj, s.d_bs, s.d_bi, FIRST_GLOBAL, d_rec.data_ptr() + 4)
    assert e.value.code == -1
    assert gpu_ctx.kernel_launches() == launches


# ---- which instantiation of eg_episode_kernel runs ----

_MANGLED = re.compile(r"eg_episode_kernelILb([01])ELi(\d)ELi(\d)E")
_DEMANGLED = re.compile(r"eg_episode_kernel<(false|true|0|1), (\d), (\d)>")


def _episode_instantiations(fn):
    """(REPLAY, GEOM, MODE) of every eg_episode_kernel launch that a CUDA profiler trace of fn() records."""
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    kernels = [e.name for e in prof.events() if str(getattr(e, "device_type", "")).endswith("CUDA")]
    if not kernels:
        pytest.skip("the CUDA profiler recorded no device kernels on this machine")
    found = set()
    for name in kernels:
        m = _MANGLED.search(name) or _DEMANGLED.search(name)
        if m:
            found.add((int(m.group(1) in ("1", "true")), int(m.group(2)), int(m.group(3))))
    return found


def test_launcher_routes_each_case_to_its_instantiation(gpu_ctx, trained):
    """Lean forms (MODE 1, MODE 2 when iterations_without_improvement > 500) run only without optional outputs and with count
    weights; everything else runs the general form (MODE 0). One call per case, on maps of each geometry (compact: the shipped
    map; medium: 101 sites of 500 m; general: 191 sites of 262 m)."""
    import os
    assets = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ireland_map")
    sx, sy, spop, ex, ey, et, ec, cx, cy = synthetic.load_ireland_arrays(assets)
    rs = np.random.RandomState(9)
    si, pi = np.sort(rs.choice(len(sx), 40, replace=False)), np.sort(rs.choice(len(ex), 12, replace=False))
    maps = {1: (sx[si].copy(), sy[si].copy(), spop[si].copy(), ex[pi].copy(), ey[pi].copy(), et[pi].copy(), ec[pi].copy(), cx, cy,
                101, 500.0),
            2: (sx, sy, spop, ex, ey, et, ec, cx, cy, 191, 262.0)}
    plain, stagnant = _with_iwi(trained, 40), _with_iwi(trained, 600)
    ctxs = {0: gpu_ctx}
    try:
        for geom, m in maps.items():
            ctxs[geom] = _lib.Context(0)
            ctxs[geom].map_set(*m)
        for geom, ctx in ctxs.items():
            assert _episode_instantiations(lambda: ctx.rollout(plain, 64, seed=3)) == {(0, geom, 1)}, geom
            assert _episode_instantiations(lambda: ctx.rollout(stagnant, 64, seed=3)) == {(0, geom, 2)}, geom
        no_counts = stagnant.clone()
        t = no_counts.table()
        t.has_count_weights = 0
        no_counts.set_table(t)
        assert _episode_instantiations(lambda: gpu_ctx.rollout(no_counts, 64, seed=3)) == {(0, 0, 0)}
        assert _episode_instantiations(lambda: gpu_ctx.rollout(stagnant, 64, seed=3, want_sites=True)) == {(0, 0, 0)}
        assert _episode_instantiations(lambda: ctxs[1].rollout(plain, 64, seed=3, want_yearly=True)) == {(0, 1, 0)}
    finally:
        for geom in maps:
            if geom in ctxs:
                ctxs[geom].close()
