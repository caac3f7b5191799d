"""Synthetic maps (BASELINE config 4): generator determinism on the CPU, and GPU parity with the oracle on maps other
than the shipped one — a coarse grid (exact one-byte nearest-plant map), a fine grid (wide instantiation: cell distances
above 254, quantised map) and the 10x scaled map itself. Same bar as test_gpu_parity.py: everything bit-exact, score within 1e-12.
"""
import os

import numpy as np
import pytest

import oracle_lib as O
from eirgrid_b200 import _abi, _lib, synthetic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ASSETS = os.path.join(ROOT, "tests", "golden", "ireland_map")
SCORE_RTOL = 1e-12


def _subset_map(n_settlements, n_plants, grid_n, step, seed):
    """A cut-down Irish map on a different candidate grid."""
    sx, sy, spop, ex, ey, et, ec, cx, cy = synthetic.load_ireland_arrays(ASSETS)
    rs = np.random.RandomState(seed)
    si = np.sort(rs.choice(len(sx), n_settlements, replace=False))
    pi = np.sort(rs.choice(len(ex), n_plants, replace=False))
    c = np.ascontiguousarray
    return (c(sx[si]), c(sy[si]), c(spop[si]), c(ex[pi]), c(ey[pi]), c(et[pi]), c(ec[pi]), cx, cy, grid_n, float(step))


def test_python_loader_equals_oracle_loader():
    a = synthetic.load_ireland_arrays(ASSETS)
    b = O.World.ireland(fast=False).arrays()
    for x, y in zip(a[:7], b):
        assert np.array_equal(x, y)
    assert len(a[7]) == 200 and len(a[8]) == 200


def test_scaled_map_is_deterministic_and_sized():
    m1 = synthetic.scaled_map(ASSETS, factor=10)
    m2 = synthetic.scaled_map(ASSETS, factor=10)
    for x, y in zip(m1, m2):
        assert np.array_equal(x, y)
    sx, sy, spop, ex, ey, et, ec, cx, cy, grid_n, step = m1
    assert len(sx) == 390 and len(ex) == 590 and grid_n == 161 and step == 312.0
    assert (grid_n - 1) * step <= 50000.0 and grid_n * grid_n >= 9.9 * 2601
    assert sx.min() >= 0 and sx.max() <= 50000 and sy.min() >= 0 and sy.max() <= 50000
    # same fuel mix as the shipped fleet (resampled with replacement): every type that occurs is a shipped one
    assert set(np.unique(et)) <= {0, 6, 7, 8, 9, 10}


def test_oracle_runs_on_a_synthetic_map():
    m = _subset_map(25, 8, 21, 2500, seed=5)
    w = O.World.from_arrays(*m)
    res, traj, sites, yearly = w.rollout(O.Weights(), 16, seed=3)
    assert (res["flags"] == 0).all() and (res["n_generators"] > 0).all()
    used = _abi.traj_row_starts(traj)[:, -1]
    placed = (np.arange(_abi.TRAJ_CAPACITY)[None, :] < used[:, None]) & (traj["actions"] < 45)
    assert sites["site"][placed].max() < 21 * 21


RESULT_FIELDS = ("net_emissions", "public_opinion", "total_cost", "power_reliability", "n_generators", "n_offsets",
                 "n_deficit_actions", "n_additional_actions", "flags")


def _assert_same_episodes(res, traj, eres, etraj):
    assert traj.tobytes() == etraj.tobytes(), "action records differ"
    for f in RESULT_FIELDS:
        assert np.array_equal(res[f], eres[f]), f
    np.testing.assert_allclose(res["score"], eres["score"], rtol=SCORE_RTOL, atol=0)


def _compare(m, n, seed):
    ctx = _lib.Context(0)
    try:
        ctx.map_set(*m)
        w = O.World.from_arrays(*m)
        res, traj, sites, yearly = ctx.rollout(_lib.Weights(), n, seed=seed, want_sites=True, want_yearly=True)
        eres, etraj, esites, eyearly = w.rollout(O.Weights(), n, seed=seed)
        _assert_same_episodes(res, traj, eres, etraj)
        assert sites.tobytes() == esites.tobytes(), "placement sites differ"
        for f in yearly["y"].dtype.names:
            if f != "reserved":
                assert np.array_equal(yearly["y"][f], eyearly["y"][f]), f
        # without sites and yearly output the launcher runs the lean instantiation of this map's geometry
        lres, ltraj, _, _ = ctx.rollout(_lib.Weights(), n, seed=seed)
        _assert_same_episodes(lres, ltraj, eres, etraj)
        # replaying the recorded actions reproduces the rollout (size-independent property)
        rres, rsites, _ = ctx.replay(traj)
        assert rsites.tobytes() == sites.tobytes()
        assert np.array_equal(rres["total_cost"], res["total_cost"]) and np.array_equal(rres["net_emissions"], res["net_emissions"])
        return res
    finally:
        ctx.close()


def _compare_lean_stagnation(m, n, seed):
    """Weights with a best strategy and iterations_without_improvement above 500, rolled out without optional outputs: the
    lean stagnation instantiation of the map's geometry against the oracle."""
    ctx = _lib.Context(0)
    try:
        ctx.map_set(*m)
        world = O.World.from_arrays(*m)
        ow, gw = O.Weights(), _lib.Weights()
        eres, etraj, _, _ = world.rollout(ow, 32, seed=seed)
        ow.update(eres, etraj)
        gw.update(eres, etraj)
        assert bytes(ow.table()) == bytes(gw.table())
        for iwi in (600, 3500):
            t = ow.table()
            t.iterations_without_improvement = iwi
            ow.set_table(t)
            gw.set_table(t)
            eres, etraj, _, _ = world.rollout(ow, n, seed=seed + iwi, want_sites=False, want_yearly=False)
            res, traj, _, _ = ctx.rollout(gw, n, seed=seed + iwi)
            # device pow() vs host pow() on a row the deficit handler edited could in principle move one draw that lands
            # exactly on a boundary (probability ~1e-13 here)
            _assert_same_episodes(res, traj, eres, etraj)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_coarse_grid_narrow_map():
    # 2.5 km cells: radii 3..12 km reach 1..4 cells; compact form of the cell distance (one IDP.4A), 21 sites per axis
    _compare(_subset_map(60, 20, 21, 2500, seed=7), 256, seed=11)


@pytest.mark.gpu
def test_odd_grid_narrow_map():
    # 47 x 47 sites of 1086 m: compact form, plant lists of every length modulo four (sentinel padding), 11-cell radius
    _compare(_subset_map(130, 59, 47, 1086, seed=8), 256, seed=12)


@pytest.mark.gpu
def test_fine_grid_wide_map():
    # 500 m cells, 101 sites per axis: 12 km = 24 cells, 1,308 table entries -> medium form (IDP.2A + add, blocks of 8 warps)
    _compare(_subset_map(40, 12, 101, 500, seed=9), 96, seed=13)


@pytest.mark.gpu
def test_more_than_128_sites_per_axis():
    # 151 sites of 331 m: medium form with coordinates above 127 (unsigned bytes) and squared norms up to 45,000 (16 bits)
    sx, sy, spop, ex, ey, et, ec, cx, cy = synthetic.load_ireland_arrays(ASSETS)
    _compare((sx, sy, spop, ex, ey, et, ec, cx, cy, 151, 331.0), 48, seed=14)


@pytest.mark.gpu
def test_more_than_181_sites_per_axis():
    # 191 sites of 262 m: squared norms no longer fit 16 bits -> general form (integer cell distances, factor table in global
    # memory, 1.0 at the end of every class)
    sx, sy, spop, ex, ey, et, ec, cx, cy = synthetic.load_ireland_arrays(ASSETS)
    _compare((sx, sy, spop, ex, ey, et, ec, cx, cy, 191, 262.0), 32, seed=16)


@pytest.mark.gpu
def test_config4_ten_times_scaled_map():
    res = _compare(synthetic.scaled_map(ASSETS, factor=10), 32, seed=15)
    assert (res["flags"] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("geometry", ["medium", "general"])
def test_lean_stagnation_instantiation(geometry):
    sx, sy, spop, ex, ey, et, ec, cx, cy = synthetic.load_ireland_arrays(ASSETS)
    if geometry == "medium":  # the map of test_fine_grid_wide_map
        _compare_lean_stagnation(_subset_map(40, 12, 101, 500, seed=9), 64, seed=17)
    else:  # the map of test_more_than_181_sites_per_axis
        _compare_lean_stagnation((sx, sy, spop, ex, ey, et, ec, cx, cy, 191, 262.0), 32, seed=18)
