"""Host side of the policy evaluation (no device needed): the record's layout against the C header, eg_eval_stats_merge against
numpy over the union of two episode sets, the JSON writer's schema, and the two command lines' argument handling."""
import ctypes as C
import json
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

import eval_ref
from eirgrid_b200 import _abi, _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ASSETS = os.path.join(ROOT, "tests", "golden", "ireland_map")
TOOL = os.path.join(ROOT, "host", "_build", "evaluate_policy")


def _random_episodes(rng, n, traj_fill=10):
    res = np.zeros(n, _abi.RESULT_DTYPE)
    res["score"] = rng.uniform(0.0, 2.0, n)
    for f in ("net_emissions", "public_opinion", "total_cost"):
        res[f] = rng.normal(1e6, 3e5, n)
    res["power_reliability"] = rng.integers(0, 2, n)
    res["n_generators"], res["n_offsets"] = rng.integers(0, 500, n), rng.integers(0, 500, n)
    res["n_deficit_actions"], res["n_additional_actions"] = rng.integers(0, 60, n), rng.integers(0, 60, n)
    res["flags"] = rng.integers(0, 16, n) * (rng.random(n) < 0.2)
    traj = np.zeros(n, _abi.TRAJ_DTYPE)
    traj["n_deficit"] = rng.integers(0, traj_fill // 2, (n, 26))
    traj["n_additional"] = rng.integers(0, traj_fill, (n, 26))
    traj["actions"] = rng.integers(0, 61, (n, _abi.TRAJ_CAPACITY))
    yearly = np.zeros(n, _abi.YEARLY_DTYPE)
    y = yearly["y"]
    y["total_population"] = rng.integers(4_000_000, 6_000_000, (n, 26))
    y["active_generators"] = rng.integers(50, 300, (n, 26))
    for f in _abi.YEAR_FIELDS[:-1]:
        y[f] = rng.normal(0.0, 1e7, (n, 26))
    y["inflation_factor"] = 1.02 ** np.arange(26)
    return res, traj, yearly


def test_record_layout_matches_the_header(tmp_path):
    """sizeof and field offsets of eg_eval_stats as the C compiler lays it out, against the ctypes structure"""
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    fields = [f[0] for f in _abi.EvalStats._fields_]
    src = tmp_path / "layout.cpp"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "eirgrid_b200.h"\nint main(void) {\n  printf("%zu\\n", sizeof(eg_eval_stats));\n'
                   + "".join('  printf("%%zu\\n", offsetof(eg_eval_stats, %s));\n' % f for f in fields)
                   + '  printf("%d\\n", EG_EVAL_COUNTER_WORDS);\n  return 0;\n}\n')
    exe = str(tmp_path / "layout")
    subprocess.run(["g++", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe], check=True)
    out = [int(v) for v in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    assert out[0] == C.sizeof(_abi.EvalStats) == 57736
    assert out[1:-1] == [getattr(_abi.EvalStats, f).offset for f in fields]
    assert out[-1] * 8 == C.sizeof(_abi.EvalStats) - _abi.EvalStats.n_flagged.offset


@pytest.mark.parametrize("yearly", [True, False])
def test_merge_matches_numpy_over_the_union(yearly):
    rng = np.random.default_rng(7)
    a = _random_episodes(rng, 3000)
    b = _random_episodes(rng, 1700)
    ya, yb = (a[2], b[2]) if yearly else (None, None)
    ra = eval_ref.reference_record(a[0], a[1], ya, first_global=100)
    rb = eval_ref.reference_record(b[0], b[1], yb, first_global=3100)
    union = eval_ref.reference_record(np.concatenate([a[0], b[0]]), np.concatenate([a[1], b[1]]),
                                      np.concatenate([ya, yb]) if yearly else None, first_global=100)
    eval_ref.assert_record_matches(ra.merge(rb), union, yearly=yearly)


def test_empty_record_is_the_identity_on_either_side():
    rng = np.random.default_rng(3)
    res, traj, yearly = _random_episodes(rng, 500)
    r = eval_ref.reference_record(res, traj, yearly, first_global=9)
    left = _abi.EvalStats().merge(r)
    right = _abi.EvalStats.from_bytes(bytes(r)).merge(_abi.EvalStats())
    assert bytes(left) == bytes(r) and bytes(right) == bytes(r)
    assert bytes(_abi.EvalStats().merge(_abi.EvalStats())) == bytes(_abi.EvalStats())


def test_equal_best_scores_keep_the_lower_id():
    rng = np.random.default_rng(5)
    res, traj, _ = _random_episodes(rng, 64)
    res["score"] = np.clip(res["score"], 0.5, 1.5)
    res["score"][10] = 1.75
    res["score"][20] = 0.25
    late = eval_ref.reference_record(res, traj, None, first_global=1000)
    early = eval_ref.reference_record(res, traj, None, first_global=0)
    m = _abi.EvalStats.from_bytes(bytes(late)).merge(early)  # shards given out of episode order
    assert (m.best_episode, m.worst_episode) == (10, 20)
    m = _abi.EvalStats.from_bytes(bytes(early)).merge(late)
    assert (m.best_episode, m.worst_episode) == (10, 20)


def test_merge_rejects_records_with_and_without_the_yearly_part():
    rng = np.random.default_rng(1)
    res, traj, yearly = _random_episodes(rng, 50)
    with pytest.raises(_lib.EirgridError) as e:
        eval_ref.reference_record(res, traj, yearly).merge(eval_ref.reference_record(res, traj, None))
    assert e.value.code == -1


def _hand_record(scores, yearly=True):
    st = _abi.EvalStats()
    st.n_episodes = len(scores)
    st.best_episode, st.worst_episode = 5, 6
    hist = st.view("score_hist")
    for s in scores:
        hist[min(int(np.floor(s * 1024.0)), 2047)] += 1
    fm = st.view("final_metrics")
    fm[0] = [np.mean(scores), ((np.asarray(scores) - np.mean(scores)) ** 2).sum(), min(scores), max(scores)]
    st.has_yearly = int(yearly)
    if yearly:
        st.view("yearly")[3, 0] = [5e6, 0.0, 5e6, 5e6]
        st.view("net_zero_or_below")[25] = len(scores)
        st.view("first_net_zero_year")[25] = len(scores)
    st.view("additional_actions")[0, 60] = 3
    st.view("deficit_actions")[2, 24] = 1
    st.n_flagged = 1
    st.view("flag_counts")[2] = 1
    return st


def test_json_schema_and_quantiles(tmp_path):
    # 100 scores: 1 at 0.0, 4 at 0.5, 90 at 1.0, 5 at exactly 2.0 (the last bin)
    scores = [0.0] + [0.5] * 4 + [1.0] * 90 + [2.0] * 5
    path = str(tmp_path / "e.json")
    _hand_record(scores).write_json(path)
    d = json.load(open(path))
    assert list(d) == ["episodes", "flagged", "final", "score_quantiles", "score_histogram", "best_episode", "worst_episode", "yearly",
                       "p_net_zero_or_below", "p_in_deficit", "first_net_zero_year", "actions"]
    assert d["episodes"] == 100 and d["flagged"] == {"any": 1, "gen_overflow": 0, "offset_overflow": 0, "record_overflow": 1, "no_site": 0}
    assert list(d["final"]) == _abi.FINAL_FIELDS
    s = d["final"]["score"]
    assert s["mean"] == np.mean(scores) and s["min"] == 0.0 and s["max"] == 2.0
    assert s["std"] == pytest.approx(np.std(scores, ddof=1), rel=1e-15)
    # lower edge of the bin holding the ceil(q n)-th score: ranks 1, 5, 25, 50, 75, 95, 99
    assert d["score_quantiles"] == {"p01": 0.0, "p05": 0.5, "p25": 1.0, "p50": 1.0, "p75": 1.0, "p95": 1.0, "p99": 2047 / 1024}
    h = d["score_histogram"]
    assert h["bin_width"] == 1 / 1024 and len(h["counts"]) == 2048 and h["out_of_range"] == 0
    assert h["counts"][0] == 1 and h["counts"][512] == 4 and h["counts"][1024] == 90 and h["counts"][2047] == 5
    assert (d["best_episode"], d["worst_episode"]) == (5, 6)
    assert list(d["yearly"]) == [str(y) for y in range(2025, 2051)]
    assert list(d["yearly"]["2028"]) == _abi.EVAL_YEAR_FIELDS
    assert d["yearly"]["2028"]["total_population"] == {"mean": 5e6, "std": 0.0, "min": 5e6, "max": 5e6}
    assert d["p_net_zero_or_below"][25] == 1.0 and d["p_net_zero_or_below"][0] == 0.0 and len(d["p_in_deficit"]) == 26
    assert d["first_net_zero_year"]["2050"] == 100 and d["first_net_zero_year"]["never"] == 0 and len(d["first_net_zero_year"]) == 27
    assert d["actions"]["2025"] == {"additional": {"DoNothing": 3}, "deficit": {}}
    assert d["actions"]["2027"] == {"additional": {}, "deficit": {_abi.action_name(24): 1}}


def test_json_single_episode_and_no_yearly(tmp_path):
    path = str(tmp_path / "one.json")
    _hand_record([1.2345], yearly=False).write_json(path)
    d = json.load(open(path))
    assert d["final"]["score"] == {"mean": 1.2345, "std": 0.0, "min": 1.2345, "max": 1.2345}
    edge = np.floor(1.2345 * 1024) / 1024
    assert set(d["score_quantiles"].values()) == {edge}
    assert d["yearly"] is None and d["p_net_zero_or_below"] is None and d["first_net_zero_year"] is None
    path = str(tmp_path / "empty.json")
    _abi.EvalStats().write_json(path)
    d = json.load(open(path))
    assert d["episodes"] == 0 and d["final"]["score"] is None and d["best_episode"] is None
    assert set(d["score_quantiles"].values()) == {None}


def _no_gpu():
    import torch
    return not torch.cuda.is_available()


def test_python_cli_rejects_malformed_arguments_and_fails_without_gpu(tmp_path):
    env = dict(os.environ, PYTHONPATH=ROOT)
    base = [sys.executable, "-m", "eirgrid_b200.evaluate"]
    for args in (["-n", "abc", "--weights", "w", "--assets", ASSETS], ["-n", "-5", "--weights", "w", "--assets", ASSETS],
                 ["--weights", "w", "--assets", ASSETS], ["-n", "5", "--weights", "w", "--assets", ASSETS, "--seed", "1.5"],
                 ["-n", "5", "--weights", "w", "--assets", ASSETS, "--nonexistent"]):
        r = subprocess.run(base + args, capture_output=True, text=True, env=env, cwd=str(tmp_path))
        assert r.returncode == 2, (args, r.stderr[-300:])
    if _no_gpu():
        w = str(tmp_path / "w.json")
        _lib.Weights().save_to_file(w)
        r = subprocess.run(base + ["-n", "16", "--weights", w, "--assets", ASSETS, "--json", str(tmp_path / "o.json")],
                           capture_output=True, text=True, env=env, cwd=str(tmp_path))
        assert r.returncode == 1 and "no CPU fallback" in r.stderr and not os.path.exists(tmp_path / "o.json")


@pytest.fixture(scope="module")
def tool():
    from eirgrid_b200 import build
    build.build()
    r = subprocess.run(["make", "-C", os.path.join(ROOT, "host")], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return TOOL


def test_host_tool_rejects_malformed_arguments_and_fails_without_gpu(tool, tmp_path):
    src = open(os.path.join(ROOT, "host", "evaluate_policy.cpp")).read()
    assert "cuda_runtime" not in src
    for args in (["-n", "abc"], ["-n", "-5"], ["-n", "99999999999999999999"], ["--devices", "x"], ["--devices", ","], ["--nonexistent"],
                 ["-n"], ["-n", "5"], ["--weights", "w", "--assets", ASSETS]):
        r = subprocess.run([tool] + args, capture_output=True, text=True)
        assert r.returncode == 2 and r.stderr.startswith("error: "), (args, r.returncode, r.stderr[:200])
    help_text = subprocess.run([tool, "--help"], capture_output=True, text=True).stdout
    for flag in ("--weights", "--assets", "-n", "--seed", "--first-episode", "--cost-only", "--no-yearly", "--json", "--devices"):
        assert flag in help_text, flag
    if _no_gpu():
        w = str(tmp_path / "w.json")
        _lib.Weights().save_to_file(w)
        r = subprocess.run([tool, "-n", "16", "--weights", w, "--assets", ASSETS], capture_output=True, text=True)
        assert r.returncode == 1 and "no CPU fallback" in r.stderr
