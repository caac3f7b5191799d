"""The small shared facts of the update rule, checked from the headers the library compiles (update_rule.hpp, eg_math.hpp):
the one Philox4x32-10 of the host and of the update kernels against the Random123 known answers, and every form of the
deficit-key order against the reference's insertion order (weights/core.rs:130-152). The harness is built with the host
compiler, so no GPU is needed."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "eirgrid_b200", "csrc")

# Random123 kat_vectors, philox4x32-10: (counter, key, output)
PHILOX_KAT = [
    ([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
    ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
    ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0], [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]),
]
# generator type of deficit keys 0..13 (GasPeaker, GasCombinedCycle, BatteryStorage, ...); key 14 is DoNothing, action code 60
DEFICIT_KEY_TYPES = [8, 7, 12, 11, 9, 0, 1, 4, 10, 5, 2, 3, 13, 14]
DO_NOTHING = 60


@pytest.fixture(scope="module")
def tables(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    exe = str(tmp_path_factory.mktemp("rule_tables") / "rule_tables")
    r = subprocess.run(["g++", "-O1", "-std=c++17", "-Wall", "-Werror", "-I" + CSRC, os.path.join(ROOT, "tests", "fuzz", "rule_tables.cpp"), "-o", exe],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    args = ["%x" % v for ctr, key, _ in PHILOX_KAT for v in ctr + key]
    out = subprocess.run([exe] + args, capture_output=True, text=True, check=True).stdout.split("\n")
    return [line.split() for line in out if line]


def test_philox_known_answers_and_uniform(tables):
    rows = [r for r in tables if r[0] == "philox"]
    assert len(rows) == len(PHILOX_KAT)
    for row, (_, _, exp) in zip(rows, PHILOX_KAT):
        assert [int(v, 16) for v in row[1:5]] == exp
        # the low 64 bits, words (0, 1), as a 53-bit uniform: exact in a double
        assert float(row[6]) == ((exp[1] << 32 | exp[0]) >> 11) * 2.0 ** -53


def test_deficit_key_order_in_every_form(tables):
    codes = [3 * t for t in DEFICIT_KEY_TYPES] + [DO_NOTHING]
    key_action = {int(r[1]): int(r[2]) for r in tables if r[0] == "key_action"}
    assert [key_action[k] for k in range(15)] == codes
    action_key = {int(r[1]): int(r[2]) for r in tables if r[0] == "action_key"}
    assert sorted(action_key) == list(range(256))
    assert action_key == {c: codes.index(c) if c in codes else -1 for c in range(256)}
    # the episode kernel's branch-free lookups: key of generator type t and type of key k, 4 bits each (0xF: CoalPlant, no key)
    key_of_type, type_of_key = (int(v, 16) for v in next(r for r in tables if r[0] == "nibbles")[1:])
    assert (key_of_type, type_of_key) == (0xDC238401F97BA65, 0xED325A4109BC78)
    assert [(key_of_type >> 4 * t) & 0xF for t in range(15)] == [DEFICIT_KEY_TYPES.index(t) if t in DEFICIT_KEY_TYPES else 0xF for t in range(15)]
    assert [(type_of_key >> 4 * k) & 0xF for k in range(14)] == DEFICIT_KEY_TYPES
