"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle on the same seeded inputs.

Bar: integer state (actions, chosen sites, counts, flags, population, reliability) bit-exact; every float of
the yearly metrics and final metrics bit-exact as well (the kernels reproduce the reference's operation order
and are compiled without FMA contraction); only `score` goes through the device's log() and is compared with
a 1e-12 relative tolerance (north_star tolerance: 1e-5).
"""
import os

import numpy as np
import pytest

import oracle_lib as O
from eirgrid_b200 import _abi, _lib

pytestmark = pytest.mark.gpu

SCORE_RTOL = 1e-12


def assert_results_equal(got, exp):
    for f in ("net_emissions", "public_opinion", "total_cost", "power_reliability"):
        assert np.array_equal(got[f], exp[f]), f
    for f in ("n_generators", "n_offsets", "n_deficit_actions", "n_additional_actions", "flags"):
        assert np.array_equal(got[f], exp[f]), f
    np.testing.assert_allclose(got["score"], exp["score"], rtol=SCORE_RTOL, atol=0)


def assert_yearly_equal(got, exp):
    for f in got["y"].dtype.names:
        if f == "reserved":
            continue
        assert np.array_equal(got["y"][f], exp["y"][f]), f


def test_site_tables_match_oracle(gpu_ctx, oracle_world):
    coast, opin = gpu_ctx.site_static()
    ocoast, oopin = oracle_world.site_static()
    assert np.array_equal(coast, ocoast)
    assert np.array_equal(opin, oopin)
    pclass_rclass = [0, 1, 1, 2, 3, 4, 5]
    pclass_water = [0, 0, 1, 1, 0, 0, 0]
    for y in (0, 7, 25):
        for pc in range(7):
            rc = pclass_rclass[pc]
            pref, stat, order = gpu_ctx.site_tables(y, rc, pc)
            opref = oracle_world.prefix(y, rc)
            assert np.array_equal(pref, opref), (y, rc)
            exp_static = opref * ocoast if pclass_water[pc] else opref.copy()
            exp_static = exp_static * (1.0 - (np.float64(np.float32(1.0)) * 0.1))
            # sorted by score descending, ties by site index ascending, and a permutation of all sites
            assert np.array_equal(np.sort(order), np.arange(len(order)))
            assert np.array_equal(stat, exp_static[order])
            key = np.lexsort((order, -stat))
            assert np.array_equal(key, np.arange(len(order)))


@pytest.mark.parametrize("seed,first", [(1, 0), (20250101, 1000)])
def test_rollout_matches_oracle_initial_weights(gpu_ctx, oracle_world, seed, first):
    n = 512
    ow = O.Weights()
    eres, etraj, esites, eyearly = oracle_world.rollout(ow, n, seed=seed, first_episode=first)
    gw = _lib.Weights()
    res, traj, sites, yearly = gpu_ctx.rollout(gw, n, seed=seed, first_episode=first, want_sites=True, want_yearly=True)
    assert traj.tobytes() == etraj.tobytes()
    assert sites.tobytes() == esites.tobytes()
    assert_results_equal(res, eres)
    assert_yearly_equal(yearly, eyearly)
    assert (res["flags"] == 0).all()


def test_replay_matches_oracle_and_rollout(gpu_ctx, oracle_world):
    n = 512
    ow = O.Weights()
    eres, etraj, esites, eyearly = oracle_world.rollout(ow, n, seed=7)
    res, sites, yearly = gpu_ctx.replay(etraj)
    assert sites.tobytes() == esites.tobytes()
    assert_results_equal(res, eres)
    assert_yearly_equal(yearly, eyearly)
    # the oracle's own replay of the same record agrees with its rollout
    rres, rtraj, rsites, ryearly = oracle_world.replay(etraj)
    assert rtraj.tobytes() == etraj.tobytes() and rsites.tobytes() == esites.tobytes()
    assert_results_equal(rres, eres)


def test_replay_edge_cases(gpu_ctx, oracle_world):
    """Empty record (deficit handler falls back to batteries), a full year of DoNothing, ragged years."""
    t = np.zeros(4, _abi.TRAJ_DTYPE)
    t[1] = _abi.pack_traj([([], [_abi.ACT_DO_NOTHING] * 20)] * 26)
    t[2] = _abi.pack_traj([([], [15, 45, 57, 40, 3] if y % 3 == 0 else []) for y in range(26)])
    t[3] = _abi.pack_traj([([24, 21], [])] + [([], [])] * 25)  # too few deficit actions: battery fallback completes the year
    res, sites, yearly = gpu_ctx.replay(t)
    eres, etraj, esites, eyearly = oracle_world.replay(t)
    assert sites.tobytes() == esites.tobytes()
    assert_results_equal(res, eres)
    assert_yearly_equal(yearly, eyearly)
    assert (res["power_reliability"] == 1.0).all()


def test_rollout_trained_weights_and_heuristic_counts(gpu_ctx, oracle_world):
    """Weights after some sequential updates (best strategy present, iwi > 0) and the loaded-file count sampler."""
    n = 256
    ow = O.Weights()
    gw = _lib.Weights()
    eres, etraj, _, _ = oracle_world.rollout(ow, 64, seed=3)
    ow.update(eres, etraj)
    gw.update(eres, etraj)
    to, tg = ow.table(), gw.table()
    assert bytes(to) == bytes(tg)
    eres, etraj, esites, eyearly = oracle_world.rollout(ow, n, seed=4)
    res, traj, sites, yearly = gpu_ctx.rollout(gw, n, seed=4, want_sites=True, want_yearly=True)
    assert traj.tobytes() == etraj.tobytes()
    assert sites.tobytes() == esites.tobytes()
    assert_results_equal(res, eres)
    tg.has_count_weights = 0
    to.has_count_weights = 0
    gw.set_table(tg)
    ow.set_table(to)
    eres, etraj, esites, _ = oracle_world.rollout(ow, n, seed=5)
    res, traj, sites, _ = gpu_ctx.rollout(gw, n, seed=5, want_sites=True)
    assert traj.tobytes() == etraj.tobytes()
    assert_results_equal(res, eres)
    # without count weights the launch without optional outputs also takes the general form
    res, traj, _, _ = gpu_ctx.rollout(gw, n, seed=5)
    assert traj.tobytes() == etraj.tobytes()
    assert_results_equal(res, eres)


def test_same_stream_quirk_q8(gpu_ctx, oracle_world):
    cfg = _abi.RunCfg(same_stream_all_episodes=1)
    gw = _lib.Weights()
    res, traj, _, _ = gpu_ctx.rollout(gw, 64, seed=12345, cfg=cfg)
    assert all(traj[i].tobytes() == traj[0].tobytes() for i in range(64))
    eres, etraj, _, _ = oracle_world.rollout(O.Weights(), 2, seed=12345, cfg=cfg)
    assert traj[0].tobytes() == etraj[0].tobytes()


def test_location_analysis_matches_oracle(gpu_ctx, oracle_world):
    for loaded in (0, 1):
        got = gpu_ctx.location_analysis(loaded)
        exp = oracle_world.location_analysis(loaded)
        assert np.array_equal(got, exp), loaded


def test_replay_best_mode_quirk_q10(gpu_ctx, oracle_world):
    """force_best_actions: the best strategy is replayed (its deficit actions are applied again as 'additional'
    actions, quirk Q10) and fallbacks are drawn when the record runs out."""
    ow = O.Weights()
    gw = _lib.Weights()
    eres, etraj, _, _ = oracle_world.rollout(ow, 48, seed=21)
    ow.update(eres, etraj)
    gw.update(eres, etraj)
    cfg = _abi.RunCfg(replay_best=1)
    eres, etraj, esites, eyearly = oracle_world.rollout(ow, 64, seed=22, cfg=cfg)
    res, traj, sites, yearly = gpu_ctx.rollout(gw, 64, seed=22, cfg=cfg, want_sites=True, want_yearly=True)
    assert traj.tobytes() == etraj.tobytes()
    assert sites.tobytes() == esites.tobytes()
    assert_results_equal(res, eres)
    assert_yearly_equal(yearly, eyearly)
    # and the update of a replay batch rebuilds the doubled records identically
    so, sg = ow.update(eres, etraj, replay=True), gw.update(res, traj, replay_best=True)
    assert bytes(ow.table()) == bytes(gw.table())
    # without a best strategy every action is a smart fallback
    eres, etraj, _, _ = oracle_world.rollout(O.Weights(), 32, seed=23, cfg=cfg)
    res, traj, _, _ = gpu_ctx.rollout(_lib.Weights(), 32, seed=23, cfg=cfg)
    assert traj.tobytes() == etraj.tobytes()
    assert_results_equal(res, eres)


def test_rollout_stagnation_branch(gpu_ctx, oracle_world):
    """iterations_without_improvement > 500: sorted, power-scaled sampling (host-tabulated for untouched rows,
    recomputed on the device for rows the deficit handler edited)."""
    ow = O.Weights()
    gw = _lib.Weights()
    eres, etraj, _, _ = oracle_world.rollout(ow, 32, seed=31)
    ow.update(eres, etraj)
    gw.update(eres, etraj)
    for iwi in (600, 3500):
        t = ow.table()
        t.iterations_without_improvement = iwi
        ow.set_table(t)
        gw.set_table(t)
        eres, etraj, esites, _ = oracle_world.rollout(ow, 256, seed=32 + iwi)
        res, traj, sites, _ = gpu_ctx.rollout(gw, 256, seed=32 + iwi, want_sites=True)
        # device pow() vs host pow() can differ in the last bit of a scaled weight: a draw landing exactly on such a
        # boundary would change one action; with 256 episodes x ~30 draws that has probability ~1e-12
        assert traj.tobytes() == etraj.tobytes()
        assert sites.tobytes() == esites.tobytes()
        assert_results_equal(res, eres)
        # the training launch (no optional outputs) runs the lean stagnation instantiation: same episodes
        res, traj, _, _ = gpu_ctx.rollout(gw, 256, seed=32 + iwi)
        assert traj.tobytes() == etraj.tobytes()
        assert_results_equal(res, eres)


def test_batch_shape_edge_cases(gpu_ctx, oracle_world):
    """Empty, single-episode and ragged batch sizes (not a multiple of the 4 warps of a block or of the grid), and a batch
    split at arbitrary points: an episode's outputs depend on (seed, episode id) only, never on the batch around it."""
    gw = _lib.Weights()
    n = 777
    res, traj, sites, yearly = gpu_ctx.rollout(gw, n, seed=55, first_episode=1000, want_sites=True, want_yearly=True)
    eres, etraj, esites, _ = oracle_world.rollout(O.Weights(), n, seed=55, first_episode=1000)
    assert traj.tobytes() == etraj.tobytes() and sites.tobytes() == esites.tobytes()
    assert_results_equal(res, eres)
    # the launch without optional outputs runs the lean instantiation of the kernel: same episodes
    rl, tl, _, _ = gpu_ctx.rollout(gw, n, seed=55, first_episode=1000)
    assert tl.tobytes() == traj.tobytes() and rl.tobytes() == res.tobytes()
    r0, t0, _, _ = gpu_ctx.rollout(gw, 0, seed=55)
    assert len(r0) == 0 and len(t0) == 0
    for first, cnt in ((0, 1), (1, 3), (4, 33), (37, 131), (168, 609)):
        r, t, s, yr = gpu_ctx.rollout(gw, cnt, seed=55, first_episode=1000 + first, want_sites=True, want_yearly=True)
        assert t.tobytes() == traj[first:first + cnt].tobytes() and s.tobytes() == sites[first:first + cnt].tobytes()
        assert r.tobytes() == res[first:first + cnt].tobytes() and yr.tobytes() == yearly[first:first + cnt].tobytes()
    rr, ss, yy = gpu_ctx.replay(traj[5:6])
    assert ss.tobytes() == sites[5:6].tobytes() and yy.tobytes() == yearly[5:6].tobytes()
    assert_results_equal(rr, res[5:6])
    r_empty, s_empty, _ = gpu_ctx.replay(traj[:0])
    assert len(r_empty) == 0


def test_location_analysis_files_match_the_shipped_cache(gpu_ctx, tmp_path):
    """eg_location_analysis_write = analyze_locations + save_cache + save_to_file (map_handler.rs:61-142,208-248,
    bin/analyze_locations.rs:19-46) on the empty map: the JSON must hold what the reference's shipped
    cache/location_analysis.json holds (frozen in tests/golden/location_analysis_scores.npz by make_location_golden.py)."""
    import json
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "location_analysis_scores.npz"))
    cache = str(tmp_path / "cache")
    txt = str(tmp_path / "location_analysis.txt")
    gpu_ctx.location_analysis_write(0, min_suitability=0.2, cache_dir=cache, text_path=txt)
    d = json.load(open(os.path.join(cache, "location_analysis.json")))
    # the shipped file predates type_to_locations (serde default on load, map_handler.rs:57-59); every other key is there
    assert sorted(k for k in d if k != "type_to_locations") == list(g["top_level_keys"])
    types = _abi.GEN_TYPES
    assert len(d["locations"]) == len(g["xy"]) == 2601
    scores = np.full((2601, 15), np.nan)
    for k, e in enumerate(d["locations"]):
        assert (e["coordinate"]["x"], e["coordinate"]["y"]) == tuple(g["xy"][k])
        for name, v in e["suitability_scores"].items():
            scores[k, types.index(name)] = v
    assert ((scores == g["scores"]) | (np.isnan(scores) & np.isnan(g["scores"]))).all()
    assert [d["type_counts"].get(t, 0) for t in types] == g["type_counts"].tolist()
    assert [d["remaining_spaces"].get(t, 0) for t in types] == g["remaining_spaces"].tolist()
    assert d["exhausted_types"] == [] and int(g["n_exhausted"]) == 0
    assert np.array_equal(np.array([[c["x"], c["y"]] for c, _ in d["multi_type_locations"]]), g["multi_xy"])
    assert [len(ts) for _, ts in d["multi_type_locations"]] == g["multi_n_types"].tolist()
    for t in types:  # type_to_locations: indices into `locations` of the entries that list the type
        idx = d["type_to_locations"].get(t, [])
        assert idx == [k for k in range(2601) if not np.isnan(scores[k, types.index(t)])]
    # serde_json's number layout: floats keep a fraction, shortest round-trip digits
    raw = open(os.path.join(cache, "location_analysis.json")).read()
    assert '"x": 24000.0' in raw and "0.5599999999999999" in raw
    report = open(txt).read().splitlines()
    assert report[0] == "Location Analysis Results" and report[3] == "Total suitable locations: 2601" and report[4] == "Multi-type locations: 2601"
    assert "Coordinate: (0, 24000)" in report and "  OffshoreWind: 0.560" in report


def test_all_sites_all_years_in_one_pass(gpu_ctx):
    """BASELINE configs[4]: every candidate site x 26 years x 15 types from one launch equals the per-year analysis of the same
    points, and a run sharded by site (8 ranks' ranges) equals the unsharded one."""
    side, step = 51, 1000.0
    full = gpu_ctx.location_analysis_sites(True, side, step)
    assert full.shape == (2601, 26, 15)
    # the candidate grid (i, j in [0, 51) x 1 km) is the non-negative quadrant of analyze_map's grid at half = 50, step = 1000
    for y in (0, 7, 25):
        ref = gpu_ctx.location_analysis(True, half_steps=50, step=step, year_index=y).reshape(101, 101, 15)[50:, 50:].reshape(2601, 15)
        assert np.array_equal(full[:, y], ref), y
    assert (full[:, 0] != full[:, 25]).any(), "population growth must move at least one decision by 2050"
    parts = [gpu_ctx.location_analysis_sites(True, side, step, first_site=r * 2601 // 8, n_sites=(r + 1) * 2601 // 8 - r * 2601 // 8) for r in range(8)]
    assert np.array_equal(np.concatenate(parts), full)
    sub = gpu_ctx.location_analysis_sites(True, side, step, year_first=3, n_years=5)
    assert np.array_equal(sub, full[:, 3:8])
    empty = gpu_ctx.location_analysis_sites(False, side, step, n_years=2)
    assert np.array_equal(empty[:, 0], empty[:, 1])  # no settlements: nothing depends on the year


def test_location_analysis_on_a_comb_coastline(oracle_world):
    """a coastline whose horizontal lines cross it up to 140 times: rows with more crossings than a crossing list holds (128)
    fall back to testing every edge; rows below the teeth use their lists. Both must equal the oracle's edge-by-edge test."""
    teeth = 70
    xs, ys = [1000.0], [1000.0]
    for k in range(teeth):  # a comb: teeth from y = 20 km up to y = 45 km, 1 km pitch
        x0 = 2000.0 + k * 650.0
        xs += [x0, x0, x0 + 300.0, x0 + 300.0]
        ys += [20000.0, 45000.0, 45000.0, 20000.0]
    xs += [49000.0, 49000.0]
    ys += [20000.0, 1000.0]
    sx, sy, spop, ex, ey, et, ec, _, _ = _ireland_arrays()
    ctx = _lib.Context(0)
    ctx.map_set(sx, sy, spop, ex, ey, et, ec, np.array(xs), np.array(ys), 51, 1000.0)
    world = O.World.from_arrays(sx, sy, spop, ex, ey, et, ec, np.array(xs), np.array(ys), 51, 1000.0, fast=False)
    for loaded in (0, 1):
        got = ctx.location_analysis(loaded)
        assert np.array_equal(got, world.location_analysis(loaded)), loaded
    # every kind of point occurs: land, water near land, open water
    marine = ctx.location_analysis(0)[:, 1]
    assert (marine == 0.0).any() and (marine == 0.8 * 0.3).any() and (marine == 0.8 * 0.7).any()
    sites = ctx.location_analysis_sites(True, 51, 1000.0, n_years=3)
    ref = ctx.location_analysis(True, half_steps=50, step=1000.0, year_index=2).reshape(101, 101, 15)[50:, 50:].reshape(2601, 15)
    assert np.array_equal(sites[:, 2], ref)
    ctx.close()


def test_suitability_rows_past_the_first_block(gpu_ctx, oracle_world):
    """A block of the suitability kernel takes one site column j and 64 consecutive i; a 1,001-site grid has 16 such chunks,
    the last one partial. Rows i on both sides of chunk boundaries, from one launch over the whole grid, against the oracle's
    analysis of the same points (site (i, j) = analysis point (i + half) * (2 half + 1) + (j + half)): year 0 and year 25
    (grown populations) on the shipped map, year 0 on the 10x map."""
    from eirgrid_b200 import synthetic
    side, half, step = 1001, 1000, 50.0
    rows = (0, 63, 64, 127, 128, 999, 1000)

    def check(ctx, world, year):
        got = ctx.location_analysis_sites(True, side, step, year_first=year, n_years=1)[:, 0].reshape(side, side, 15)
        for i in rows:
            exp = world.location_analysis(True, half=half, step=step, first=(i + half) * (2 * half + 1) + half, n=side)
            assert np.array_equal(got[i], exp), (year, i)

    check(gpu_ctx, oracle_world, 0)
    sx, sy, spop, ex, ey, et, ec, cx, cy = _ireland_arrays()
    pop = spop.astype(np.float64)
    for _ in range(25):
        pop = np.floor(pop * 1.01 + 0.5)  # f64::round of positive values
    check(gpu_ctx, O.World.from_arrays(sx, sy, pop.astype(np.uint32), ex, ey, et, ec, cx, cy, 51, 1000.0, fast=False), 25)
    m = synthetic.scaled_map(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ireland_map"), 10)
    ctx = _lib.Context(0)
    try:
        ctx.map_set(*m)
        check(ctx, O.World.from_arrays(*m, fast=False), 0)
    finally:
        ctx.close()


def _ireland_arrays():
    from eirgrid_b200 import synthetic
    return synthetic.load_ireland_arrays(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ireland_map"))
