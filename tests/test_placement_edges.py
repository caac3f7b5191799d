"""The placement walk (Warp::place in csrc/episode.cu, walking the lists eg_site_rank_kernel in csrc/site_tables.cu sorts) against
the oracle where the shipped and synthetic maps never take it: exact ties, zero and subnormal scores, searches that find no site,
and the edges of each form of the cell-distance arithmetic.

The reference keeps the first strict maximum in scan order. The kernel reproduces that rule three times: the rank sort orders equal
static scores by site index, a walk step takes the lowest cell among its equal maxima, and a later step replaces the best so far
only with a higher score or an equal score at a lower cell. On the shipped map no two site scores are equal and none is 0, so those
rules never decide an output there. The maps of this file are built so that they do:

- symmetric: one settlement on the centre cell of an odd grid, no existing plants, the coastline at the four corners. Mirror sites
  have bit-identical scores (41 x 41 at 1,000 m has 198 distinct prefix values for 1,681 sites), in all three forms.
- underflowing: ~440 settlements in one 8 km corner. The settlement product underflows: hundreds of sites score exactly 0 and
  hundreds are subnormal.
- tiny: the Irish data on 2 x 2, 3 x 3 and 5 x 5 sites. Lists shorter than one walk step; the grid fills up and searches find no
  site (EG_FLAG_NO_SITE) in the deficit loop and in the additional actions.
- form limits: the Irish data at 64 / 65, 181 / 182 and 255 sites per axis (the largest grid eg_map_set accepts), and the medium
  and general forms picked by the size of the factor table on small grids (64 at 300 m, 40 at 150 m). tests/test_host_tables.py
  pins which form each of these griddings gets.

Bar of test_synthetic_maps.py: action records and sites byte-identical, results and every yearly field bit-exact, score within
1e-12; each rollout is repeated without outputs (lean instantiation) and replayed.
"""
import os

import numpy as np
import pytest

import oracle_lib as O
from eirgrid_b200 import _abi, _lib, synthetic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ASSETS = os.path.join(ROOT, "tests", "golden", "ireland_map")
SCORE_RTOL = 1e-12
WALK_STEP = 32                                                     # candidate sites per step of the walk (one per lane)
RADII = [3000.0, 5000.0, 6000.0, 7000.0, 8000.0, 12000.0]           # by radius class
PCLASS_OF_TYPE = [1, 2, 0, 0, 0, 6, 5, 5, 0, 0, 4, 4, 0, 3, 3]     # csrc/host_tables.cpp
RCLASS_OF_PCLASS = [0, 1, 1, 2, 3, 4, 5]
WATER_OF_PCLASS = [0, 0, 1, 1, 0, 0, 0]
SIZE_FACTOR = 1.0 - float(np.float32(1.0)) * 0.1                  # 1 - size_penalty * 0.1 with the f32 size penalty
WATER_TYPES = (1, 13, 14)                                          # OffshoreWind, TidalGenerator, WaveEnergy
RESULT_FIELDS = ("net_emissions", "public_opinion", "total_cost", "power_reliability", "n_generators", "n_offsets",
                 "n_deficit_actions", "n_additional_actions", "flags")


# ---- maps ---------------------------------------------------------------------------------------------------------------------

def _symmetric_map(n, step):
    """One settlement on the centre cell, no existing plants, coastline points at the four corners of the grid: the scores are
    invariant under the eight symmetries of the square, bit for bit (x - c and c - x square to the same double)."""
    c, far = (n - 1) // 2 * step, (n - 1) * step
    none = np.zeros(0)
    return (np.array([c]), np.array([c]), np.array([600000], np.uint32), none, none, np.zeros(0, np.uint8), none,
            np.array([0.0, 0.0, far, far]), np.array([0.0, far, 0.0, far]), n, float(step))


def _underflow_map(seed=0, n_settlements=440):
    """The Irish plants and coastline, with ~440 settlements in the 8 km corner at the origin: far from the corner the product of
    440 factors (1 + pop/1e6) / (1 + d/1e4) leaves the double range."""
    _, _, _, ex, ey, et, ec, cx, cy = synthetic.load_ireland_arrays(ASSETS)
    rs = np.random.RandomState(seed)
    sx, sy = rs.uniform(0.0, 8000.0, n_settlements), rs.uniform(0.0, 8000.0, n_settlements)
    spop = rs.randint(2000, 20000, n_settlements).astype(np.uint32)
    return (sx, sy, spop, ex, ey, et, ec, cx, cy, 51, 1000.0)


def _irish_map(n, step):
    return tuple(synthetic.load_ireland_arrays(ASSETS)) + (n, float(step))


MAPS = {
    "symmetric_compact_41x1000": lambda: _symmetric_map(41, 1000),
    "symmetric_medium_101x500": lambda: _symmetric_map(101, 500),
    "symmetric_general_41x150": lambda: _symmetric_map(41, 150),
    "underflow_51x1000": lambda: _underflow_map(),
    "tiny_2x1000": lambda: _irish_map(2, 1000),
    "tiny_3x1000": lambda: _irish_map(3, 1000),
    "tiny_5x1000": lambda: _irish_map(5, 1000),
    "compact_limit_64x790": lambda: _irish_map(64, 790),
    "medium_65x780": lambda: _irish_map(65, 780),
    "medium_limit_181x277": lambda: _irish_map(181, 277),
    "general_182x275": lambda: _irish_map(182, 275),
    "general_limit_255x196": lambda: _irish_map(255, 196),
    "medium_by_table_64x300": lambda: _irish_map(64, 300),
    "general_by_table_40x150": lambda: _irish_map(40, 150),
}
SYMMETRIC = [k for k in MAPS if k.startswith("symmetric")]
TINY = [k for k in MAPS if k.startswith("tiny")]
SCORED = SYMMETRIC + ["underflow_51x1000"] + TINY   # maps small enough for the numpy re-evaluation of every placement


def _episodes(name):
    """episodes per rollout: the oracle's placement search scans every site"""
    n = MAPS[name]()[9]
    return 16 if n > 150 else 64


_worlds = {}


def _world(name):
    if name not in _worlds:
        _worlds[name] = O.World.from_arrays(*MAPS[name]())
    return _worlds[name]


# ---- numpy reference of the placement search -----------------------------------------------------------------------------------

def _type_class(t):
    pc = PCLASS_OF_TYPE[t]
    return pc, RCLASS_OF_PCLASS[pc], bool(WATER_OF_PCLASS[pc])


class _Search:
    """find_suitable_location restated in numpy on one map: the prefix of the site (settlements and existing plants, from the
    oracle's tables), the factor distance / radius of every plant the episode built within the radius, in plant order, then the
    coastline factor and the size factor. Also the walk order of the kernel: static score descending, site index ascending."""

    def __init__(self, name):
        m = MAPS[name]()
        self.world = _world(name)
        self.n, self.step = m[9], m[10]
        site = np.arange(self.n * self.n)
        self.x, self.y = (site // self.n) * self.step, (site % self.n) * self.step
        self.coast = self.world.site_static()[0]
        self._prefix = {}

    def prefix(self, y, rc):
        if (y, rc) not in self._prefix:
            self._prefix[(y, rc)] = self.world.prefix(y, rc)
        return self._prefix[(y, rc)]

    def static(self, t, y):
        _, rc, water = _type_class(t)
        s = self.prefix(y, rc)
        return (s * self.coast if water else s) * SIZE_FACTOR

    def scores(self, t, y, plants):
        _, rc, water = _type_class(t)
        r = RADII[rc]
        sc = self.prefix(y, rc).copy()
        for px, py in plants:
            dx, dy = self.x - px, self.y - py
            d = np.sqrt(dx * dx + dy * dy)
            inside = d < r
            sc[inside] = sc[inside] * (d[inside] / r)
        if water:
            sc = sc * self.coast
        return sc * SIZE_FACTOR

    def walk_order(self, t, y):
        st = self.static(t, y)
        return np.lexsort((np.arange(len(st)), -st))


def _replay_placements(search, rec, sites):
    """Re-evaluates every placement of one recorded episode in the reference's order. Returns one tuple per placement:
    (type, year, site found by numpy or -1, number of sites at the best score, tie across walk steps with the lower cell later)."""
    out = []
    plants = []
    for y, (rows, srows) in enumerate(zip(_abi.traj_rows(rec), _abi.traj_rows(rec, sites))):
        for acts, ss in zip(rows, srows):
            for a, s in zip(acts.tolist(), ss.tolist()):
                if a >= 45:
                    continue
                t = a // 3
                sc = search.scores(t, y, plants)
                best = sc.max()
                found = int(np.argmax(sc)) if best > 0.0 else -1
                tied = np.nonzero(sc == best)[0] if best > 0.0 else np.zeros(0, np.int64)
                later_lower = False
                if len(tied) > 1:
                    pos = np.empty(len(sc), np.int64)
                    pos[search.walk_order(t, y)] = np.arange(len(sc))
                    first_step = pos[tied].min() // WALK_STEP
                    later_lower = bool((pos[tied[0]] // WALK_STEP) > first_step)   # the lowest tied cell sits in a later step
                out.append((t, y, found, s, len(tied), later_lower))
                if found >= 0:
                    plants.append((search.x[found], search.y[found]))
    return out


# ---- CPU tests: the oracle as the reference, and what each map exercises --------------------------------------------------------

@pytest.mark.parametrize("name", list(MAPS))
def test_oracle_fast_and_faithful_agree(name):
    """FAST (tabulated prefix, the mode the GPU tests compare with) against FAITHFUL (every product recomputed per search)."""
    w = _world(name)
    faithful = O.World.from_arrays(*MAPS[name](), fast=False)
    n = 4 if MAPS[name]()[9] > 150 else 24
    res, traj, sites, yearly = w.rollout(O.Weights(), n, seed=5)
    fres, ftraj, fsites, fyearly = faithful.rollout(O.Weights(), n, seed=5, mode=O.FAITHFUL)
    assert traj.tobytes() == ftraj.tobytes()
    assert sites.tobytes() == fsites.tobytes()
    assert res.tobytes() == fres.tobytes()


@pytest.mark.parametrize("name", SCORED)
def test_numpy_search_reproduces_the_oracle(name):
    """The numpy restatement finds the oracle's site for every placement (SITE_NONE when every score is 0)."""
    search = _Search(name)
    res, traj, sites, _ = _world(name).rollout(O.Weights(), 8, seed=9)
    for e in range(len(res)):
        for t, y, found, got, _, _ in _replay_placements(search, traj[e], sites["site"][e]):
            assert got == (found if found >= 0 else _abi.SITE_NONE), (e, t, y)


@pytest.mark.parametrize("name", SYMMETRIC)
def test_symmetric_maps_decide_placements_among_ties(name):
    search = _Search(name)
    pre = search.prefix(0, 0)
    assert len(np.unique(pre)) < len(pre) // 5
    if name == "symmetric_compact_41x1000":
        assert len(np.unique(pre)) == 198
    res, traj, sites, _ = _world(name).rollout(O.Weights(), 16, seed=11)
    placements = [p for e in range(len(res)) for p in _replay_placements(search, traj[e], sites["site"][e])]
    tied = [p for p in placements if p[4] >= 2]
    # a good part of the placements are decided among mirror images (40 % to 70 % on these maps), water types among them
    assert len(tied) > len(placements) // 4
    assert any(p[0] in WATER_TYPES for p in tied)
    # mirror sites have equal static scores, so the rank sort lists them by index and the lowest cell always comes first: the
    # cross-step clause of the walk (an equal score at a lower cell in a later step) is never what decides a placement here
    assert not any(p[5] for p in placements)


def test_underflowing_map_has_zero_and_subnormal_scores():
    search = _Search("underflow_51x1000")
    tiny = np.finfo(np.float64).tiny
    for y in (0, 25):
        for rc in range(6):
            pre = search.prefix(y, rc)
            assert (pre == 0.0).sum() > 300 and ((pre > 0.0) & (pre < tiny)).sum() > 200, (y, rc)
    # static scores too, for a land and a water class
    for t in (5, 13):
        st = search.static(t, 0)
        assert (st == 0.0).sum() > 300 and ((st > 0.0) & (st < tiny)).sum() > 200
    res, _, _, _ = _world("underflow_51x1000").rollout(O.Weights(), 16, seed=3)
    assert (res["n_generators"] > 0).all()


def _no_site_events(res, traj, sites, yearly):
    """(episodes whose deficit loop ran out of sites, episodes with an additional placement that found no site).
    The deficit loop leaves with the year still short of power only when a search finds no site (the plant list cannot fill on
    these maps), and nothing later in the year lowers the balance: a year that ends below 0 had such a search. An additional
    placement without a site is recorded with SITE_NONE."""
    deficit = (yearly["y"]["power_balance"] < 0.0).any(axis=1)
    additional = np.zeros(len(res), bool)
    for e in range(len(res)):
        for (_, acts), (_, ss) in zip(_abi.traj_rows(traj[e]), _abi.traj_rows(traj[e], sites["site"][e])):
            additional[e] |= bool(((acts < 45) & (ss == _abi.SITE_NONE)).any())
    return deficit, additional


@pytest.mark.parametrize("name", TINY)
def test_tiny_maps_run_out_of_sites(name):
    res, traj, sites, yearly = _world(name).rollout(O.Weights(), 64, seed=3)
    flagged = (res["flags"] & _abi.FLAG_NO_SITE) != 0
    assert np.isin(res["flags"], (0, _abi.FLAG_NO_SITE)).all()
    deficit, additional = _no_site_events(res, traj, sites, yearly)
    assert np.array_equal(flagged, deficit | additional)
    if name == "tiny_5x1000":
        assert flagged.any() and not flagged.all()
    else:
        assert flagged.all()
    if name == "tiny_2x1000":
        assert deficit.any() and additional.any()


# ---- GPU tests: kernel against oracle -----------------------------------------------------------------------------------------

def _assert_same_episodes(res, traj, eres, etraj):
    assert traj.tobytes() == etraj.tobytes(), "action records differ"
    for f in RESULT_FIELDS:
        assert np.array_equal(res[f], eres[f]), f
    np.testing.assert_allclose(res["score"], eres["score"], rtol=SCORE_RTOL, atol=0)


def _assert_same_yearly(yearly, eyearly):
    for f in yearly["y"].dtype.names:
        if f != "reserved":
            assert np.array_equal(yearly["y"][f], eyearly["y"][f]), f


@pytest.fixture(scope="module")
def ctxs():
    """one context per map, created on first use"""
    made = {}

    def get(name):
        if name not in made:
            ctx = _lib.Context(0)
            ctx.map_set(*MAPS[name]())
            made[name] = ctx
        return made[name]

    yield get
    for ctx in made.values():
        ctx.close()


def _rollout_parity(ctx, world, gw, ow, n, seed, cfg=None):
    """rollout with sites and yearly rows, the lean rollout, and the replay of the record, against the oracle"""
    eres, etraj, esites, eyearly = world.rollout(ow, n, seed=seed, cfg=cfg)
    res, traj, sites, yearly = ctx.rollout(gw, n, seed=seed, cfg=cfg, want_sites=True, want_yearly=True)
    _assert_same_episodes(res, traj, eres, etraj)
    assert sites.tobytes() == esites.tobytes(), "placement sites differ"
    _assert_same_yearly(yearly, eyearly)
    lres, ltraj, _, _ = ctx.rollout(gw, n, seed=seed, cfg=cfg)
    _assert_same_episodes(lres, ltraj, eres, etraj)
    rres, rsites, ryearly = ctx.replay(traj, cfg=cfg)
    assert rsites.tobytes() == sites.tobytes()
    for f in ("net_emissions", "total_cost", "flags"):
        assert np.array_equal(rres[f], res[f]), f
    return eres


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MAPS))
def test_rollout_initial_weights(ctxs, name):
    eres = _rollout_parity(ctxs(name), _world(name), _lib.Weights(), O.Weights(), _episodes(name), seed=21)
    if name.startswith("tiny") and name != "tiny_5x1000":
        assert (eres["flags"] & _abi.FLAG_NO_SITE).all()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MAPS))
def test_rollout_trained_table_with_stagnation(ctxs, name):
    """Weights after one update (a best strategy), then iterations_without_improvement above 500: the stagnation sampler, in the
    rollout with outputs and in the lean instantiation."""
    ctx, world = ctxs(name), _world(name)
    ow, gw = O.Weights(), _lib.Weights()
    eres, etraj, _, _ = world.rollout(ow, 32, seed=22)
    ow.update(eres, etraj)
    gw.update(eres, etraj)
    assert bytes(ow.table()) == bytes(gw.table())
    for iwi in (600, 3500):
        t = ow.table()
        t.iterations_without_improvement = iwi
        ow.set_table(t)
        gw.set_table(t)
        _rollout_parity(ctx, world, gw, ow, _episodes(name) // 2, seed=23 + iwi)


@pytest.mark.gpu
def test_rollout_cost_only_mode(ctxs):
    name = "symmetric_compact_41x1000"
    cfg = _abi.RunCfg(cost_only=1)
    ow, gw = O.Weights(), _lib.Weights()
    eres, etraj, _, _ = _world(name).rollout(ow, 32, seed=24, cfg=cfg)
    ow.update(eres, etraj)
    gw.update(eres, etraj)
    _rollout_parity(ctxs(name), _world(name), gw, ow, 64, seed=25, cfg=cfg)


ADVERSARIAL_TYPES = [1, 13, 14, 5, 6, 10, 0, 12, 2, 11]   # the water types first, then one of every radius class


def _adversarial_records(seed, n):
    """Records that place 12 to 18 plants a year, most of one chosen type per episode, with a few deficit actions and offsets."""
    rs = np.random.RandomState(seed)
    t = np.zeros(n, _abi.TRAJ_DTYPE)
    for e in range(n):
        main = ADVERSARIAL_TYPES[e % len(ADVERSARIAL_TYPES)]
        rows = []
        for y in range(26):
            nd = rs.randint(0, 3)
            na = rs.randint(12, 19)
            acts = 3 * main + rs.randint(0, 3, nd + na)
            other = rs.rand(nd + na) < 0.2
            acts[other] = rs.randint(0, 61, other.sum())
            rows.append((acts[:nd], acts[nd:]))
        t[e] = _abi.pack_traj(rows)
    return t


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(MAPS))
def test_replay_adversarial_records(ctxs, name):
    n = 10 if MAPS[name]()[9] > 150 else 30
    t = _adversarial_records(31, n)
    eres, etraj, esites, eyearly = _world(name).replay(t)
    assert (eres["n_generators"] <= 560).all() and (eres["n_offsets"] <= 520).all()   # within the device's plant and offset lists
    res, sites, yearly = ctxs(name).replay(t)
    assert sites.tobytes() == esites.tobytes(), "placement sites differ"
    for f in RESULT_FIELDS:
        assert np.array_equal(res[f], eres[f]), f
    np.testing.assert_allclose(res["score"], eres["score"], rtol=SCORE_RTOL, atol=0)
    _assert_same_yearly(yearly, eyearly)


@pytest.mark.gpu
@pytest.mark.parametrize("name", SCORED)
def test_site_tables_against_oracle(ctxs, name):
    """eg_map_site_tables: prefix and static scores bit-exact, the walk list sorted by static score with equal scores by index."""
    ctx, world = ctxs(name), _world(name)
    coast, opinion = ctx.site_static()
    ocoast, oopinion = world.site_static()
    assert np.array_equal(coast, ocoast) and np.array_equal(opinion, oopinion)
    ties = 0
    for y in (0, 13, 25):
        for pc in range(7):
            rc = RCLASS_OF_PCLASS[pc]
            pref, stat, order = ctx.site_tables(y, rc, pc)
            opref = world.prefix(y, rc)
            assert np.array_equal(pref, opref), (y, rc)
            exp_static = (opref * ocoast if WATER_OF_PCLASS[pc] else opref) * SIZE_FACTOR
            assert np.array_equal(order.astype(np.int64), np.lexsort((np.arange(len(order)), -exp_static))), (y, pc)
            assert np.array_equal(stat, exp_static[order])
            ties += int((np.diff(stat) == 0.0).sum())
    if name not in TINY:   # mirror sites, and the sites whose product underflowed to 0
        assert ties > 0


def _stats_flagged(ctx, w, res, traj):
    """the statistics kernel's count of flagged episodes (word 2 of the statistics table)"""
    import torch
    dev = torch.device("cuda", 0)
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).to(dev)
    d_res, d_traj = up(res), up(traj)
    d_stats = torch.zeros(_abi.STATS_WORDS, dtype=torch.int64, device=dev)
    d_bs = torch.zeros(1, dtype=torch.float64, device=dev)
    d_bi = torch.zeros(1, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    ctx.weights_upload(w)
    ctx.update_stats_device(w, len(res), d_res, d_traj, d_stats, d_bs, d_bi)
    ctx.sync()
    return int(d_stats.cpu().numpy()[2])


@pytest.mark.gpu
def test_no_site_counts_downstream(ctxs):
    """On the 5 x 5 map some episodes run out of sites: the statistics kernel, eg_evaluate and the host update count exactly the
    oracle's flagged episodes."""
    name = "tiny_5x1000"
    ctx, world = ctxs(name), _world(name)
    n, seed = 512, 41
    eres, etraj, _, _ = world.rollout(O.Weights(), n, seed=seed)
    no_site = int(((eres["flags"] & _abi.FLAG_NO_SITE) != 0).sum())
    flagged = int((eres["flags"] != 0).sum())
    assert flagged == no_site and 0 < no_site < n
    gw = _lib.Weights()
    res, traj, _, _ = ctx.rollout(gw, n, seed=seed)
    _assert_same_episodes(res, traj, eres, etraj)
    assert _stats_flagged(ctx, gw, res, traj) == flagged
    st = ctx.evaluate(gw, n, seed=seed)
    assert st.n_episodes == n and st.n_flagged == flagged
    assert list(st.flag_counts) == [int(((eres["flags"] >> b) & 1).sum()) for b in range(_abi.EVAL_N_FLAGS)]
    assert st.flag_counts[3] == no_site                                  # bit 3: EG_FLAG_NO_SITE
    assert gw.update(res, traj).n_flagged == flagged
