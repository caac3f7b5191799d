"""The host-built tables the episode kernel's placement walk relies on (csrc/host_tables.cpp), on the CPU.

The kernel's evaluation loop has no range test: a plant out of range must read a factor of exactly 1.0 at index r2_limit of its
radius class — in the block-shared copy of the table (one extra entry per class, hence the offsets) and in the global table (row
stride above the largest limit). It picks the form of its cell-distance arithmetic from `near_geom`, and reads one packed word
per type. This test pins all of that for the shipped map and for re-gridded versions of it, with the harness built under
ASan + UBSan like the other host harnesses.
"""
import math
import os
import re

import pytest

from test_host_sanitizers import ASSETS, _build, _run

RADII = [3000.0, 5000.0, 6000.0, 7000.0, 8000.0, 12000.0]          # metal_location_search.rs:139-146, by radius class
MAPS = [(51, 1000.0, 0), (21, 2500.0, 0), (47, 1086.0, 0), (64, 790.0, 0), (65, 780.0, 1), (101, 500.0, 1), (151, 331.0, 1),
        (161, 312.0, 1), (181, 277.0, 1), (182, 275.0, 2), (191, 262.0, 2),
        # the griddings of test_placement_edges.py: lists shorter than one walk step, the largest grid eg_map_set accepts, and the
        # medium and general forms chosen by the size of the factor table on grids small enough for a narrower one
        (2, 1000.0, 0), (3, 1000.0, 0), (5, 1000.0, 0), (41, 1000.0, 0), (255, 196.0, 2), (64, 300.0, 1), (40, 150.0, 2),
        (41, 150.0, 2)]


def _limits(step):
    out = []
    for r in RADII:
        d2 = 0
        while math.sqrt(d2 * step * step) < r:
            d2 += 1
        out.append(d2)
    return out


@pytest.fixture(scope="module")
def dump(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("host_tables")
    exe = _build(tmp, "host_tables_dump.cpp", "host_tables.cpp")
    args = [os.path.join(ASSETS, f) for f in ("settlements.json", "ireland_generators.csv", "coastline_points.json")]
    for n, step, _ in MAPS:
        args += [str(n), repr(step)]
    text = _run(exe, args, str(tmp))
    maps = {}
    cur = None
    for line in text.splitlines():
        m = re.match(r"map (\d+) (\S+) geom=(\d+) stride=(\d+) entries=(\d+)", line)
        if m:
            cur = dict(geom=int(m.group(3)), stride=int(m.group(4)), entries=int(m.group(5)), rclass=[], types=[])
            maps[(int(m.group(1)), float(m.group(2)))] = cur
            continue
        m = re.match(r"\s+rclass (\d+) limit=(\d+) offset=(\d+) first=(\S+) last_inside=(\S+) at_limit=(\S+)", line)
        if m:
            cur["rclass"].append(dict(limit=int(m.group(2)), offset=int(m.group(3)), first=float(m.group(4)), last=float(m.group(5)),
                                      at_limit=float(m.group(6))))
            continue
        m = re.match(r"\s+type (\d+) sums=(\S+) net_mw=(\S+) co2=(\S+) acc=(\d) info=(\d+),(\d+) pclass=(\d+) rclass=(\d+) water=(\d)", line)
        if m:
            cur["types"].append(dict(sums=[float(x) for x in m.group(2).split(",")], net_mw=float(m.group(3)), co2=float(m.group(4)),
                                     acc=int(m.group(5)), info=(int(m.group(6)), int(m.group(7))), pclass=int(m.group(8)),
                                     rclass=int(m.group(9)), water=int(m.group(10))))
    return maps


def test_every_map_was_built(dump):
    assert sorted(dump) == sorted((n, step) for n, step, _ in MAPS)


@pytest.mark.parametrize("n,step,geom", MAPS)
def test_geometry_and_factor_table_layout(dump, n, step, geom):
    d = dump[(n, step)]
    limits = _limits(step)
    assert [r["limit"] for r in d["rclass"]] == limits
    # block-shared copy: every class is followed by one entry (the 1.0), the offsets are running sums of limit + 1
    off = 0
    for r in d["rclass"]:
        assert r["offset"] == off
        off += r["limit"] + 1
    assert d["entries"] == off == sum(limits) + 6
    # global table: the row of a class is longer than its limit, and the entry at the limit is exactly 1.0
    assert d["stride"] == max(limits) + 1
    for r, radius in zip(d["rclass"], RADII):
        assert r["first"] == 0.0                      # a plant on the site itself: distance 0
        assert 0.0 < r["last"] < 1.0                  # inside the radius: distance / radius < 1
        assert r["at_limit"] == 1.0
    # the form of the cell-distance arithmetic: compact up to 64 sites per axis (and a table of at most 2048 entries), medium up to
    # 181 (|g|^2 < 65536; at most 5600 entries), general beyond
    assert d["geom"] == geom
    if geom == 0:
        assert n <= 64 and d["entries"] <= 2048
    elif geom == 1:
        assert n <= 181 and d["entries"] <= 5600 and 2 * (n - 1) ** 2 < 65536


def test_per_type_words_agree_with_the_tables_they_replace(dump):
    for d in dump.values():
        assert len(d["types"]) == 15
        for t in d["types"]:
            # (plain, intermittent, storage, CO2): the net output in the slot of the accumulator class, +0.0 elsewhere
            want = [0.0, 0.0, 0.0, t["co2"]]
            want[t["acc"]] = t["net_mw"]
            assert t["sums"] == want
            x, y = t["info"]
            assert x & 0xF == t["pclass"] and (x >> 4) & 0xF == t["rclass"] and (x >> 8) & 1 == t["water"]
            assert y == d["rclass"][t["rclass"]]["limit"]
            if d["geom"] != 2:   # first entry of the class in the block-shared table (16 bits)
                assert x >> 16 == d["rclass"][t["rclass"]]["offset"]
