"""Policy evaluation on the GPU (eg_evaluate, eg_eval_accumulate_device; csrc/evaluate.cu) against a numpy reduction of the same
episodes copied out with ctx.rollout, its determinism contract, hand-built inputs, errors, and the two command lines."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import eval_ref
import oracle_lib as O
from eirgrid_b200 import _abi, _lib, synthetic

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ASSETS = os.path.join(ROOT, "tests", "golden", "ireland_map")
N = 65536 + 4097  # two chunks, the second ragged
FIRST = 123457
SIZE = C.sizeof(_abi.EvalStats)


def _torch():
    import torch
    return torch


@pytest.fixture(scope="module")
def trained(oracle_world):
    """Weights with a best strategy (one oracle batch and one update)."""
    w = _lib.Weights()
    res, traj, _, _ = oracle_world.rollout(O.Weights(), 32, seed=41)
    w.update(res, traj)
    assert w.table().has_best
    return w


def _parts(st, yearly):
    """bytes of the parts that do not depend on with_yearly: final moments, best/worst, histogram, flags, actions"""
    b = bytes(st)
    fm = _abi.EvalStats.final_metrics
    out = b[_abi.EvalStats.best_episode.offset:_abi.EvalStats.has_yearly.offset] + b[fm.offset:fm.offset + fm.size]
    out += b[_abi.EvalStats.n_flagged.offset:_abi.EvalStats.net_zero_or_below.offset] + b[_abi.EvalStats.additional_actions.offset:]
    return out


@pytest.mark.parametrize("which", ["initial", "trained"])
def test_evaluate_matches_numpy_reduction_and_is_bit_stable(gpu_ctx, trained, which):
    w = _lib.Weights() if which == "initial" else trained
    res, traj, _, yearly = gpu_ctx.rollout(w, N, seed=3, first_episode=FIRST, want_yearly=True)
    ref_y = eval_ref.reference_record(res, traj, yearly, first_global=FIRST)
    ref_n = eval_ref.reference_record(res, traj, None, first_global=FIRST)
    del yearly
    got_y = gpu_ctx.evaluate(w, N, seed=3, first_episode=FIRST, with_yearly=True)
    got_n = gpu_ctx.evaluate(w, N, seed=3, first_episode=FIRST, with_yearly=False)
    eval_ref.assert_record_matches(got_y, ref_y, yearly=True)
    eval_ref.assert_record_matches(got_n, ref_n, yearly=False)
    assert got_n.has_yearly == 0 and not got_n.view("yearly").any()
    # bit stability: a repeated call, the yearly-independent parts of both modes, a call after unrelated rollouts
    assert bytes(gpu_ctx.evaluate(w, N, seed=3, first_episode=FIRST, with_yearly=True)) == bytes(got_y)
    assert _parts(got_y, True) == _parts(got_n, False)
    gpu_ctx.rollout(trained, 3000, seed=99, first_episode=7, want_sites=True, want_yearly=True)
    assert bytes(gpu_ctx.evaluate(w, N, seed=3, first_episode=FIRST, with_yearly=False)) == bytes(got_n)
    # fields that no action changes: every episode has the same value, m2 is exactly 0
    one = gpu_ctx.rollout(w, 1, seed=3, first_episode=FIRST, want_yearly=True)[3]
    for f in ("total_population", "total_power_usage", "inflation_factor"):
        m = got_y.view("yearly")[:, _abi.EVAL_YEAR_FIELDS.index(f)]
        assert np.array_equal(m[:, 1], np.zeros(26)), f
        assert np.array_equal(m[:, 0], one["y"][f][0].astype(np.float64)), f
    # the best episode, rolled out alone, gives the recorded maximum
    best = gpu_ctx.rollout(w, 1, seed=3, first_episode=got_y.best_episode)[0]
    assert best["score"][0] == got_y.view("final_metrics")[0, 3]


def test_split_and_merge_equals_one_range(gpu_ctx, trained):
    whole = gpu_ctx.evaluate(trained, N, seed=5, first_episode=FIRST)
    a = 30001
    merged = gpu_ctx.evaluate(trained, a, seed=5, first_episode=FIRST).merge(gpu_ctx.evaluate(trained, N - a, seed=5, first_episode=FIRST + a))
    assert eval_ref.counter_bytes(merged) == eval_ref.counter_bytes(whole)
    eval_ref.assert_record_matches(merged, whole, yearly=True)


def _accumulate(ctx, res, traj, yearly, first, d_acc=None):
    torch = _torch()
    dev = torch.device("cuda", 0)
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).to(dev)
    if d_acc is None:
        d_acc = torch.zeros(SIZE, dtype=torch.uint8, device=dev)
    d_res, d_traj = up(res), up(traj)
    d_y = up(yearly) if yearly is not None else None
    torch.cuda.synchronize()
    ctx.eval_accumulate_device(len(res), d_res, d_traj, d_y, first, d_acc)
    ctx.sync()
    return _abi.EvalStats.from_bytes(d_acc.cpu().numpy().tobytes()), d_acc


def test_hand_built_inputs(gpu_ctx, trained):
    res, traj, _, yearly = gpu_ctx.rollout(trained, 700, seed=8, want_yearly=True)
    special = [0.0, 2.0, -0.25, 2.5, np.nan, 1.0 / 1024, 2047.0 / 1024]
    res["score"][[3, 50, 51, 300, 301, 400, 401]] = special
    res["flags"][:16] = np.arange(16)  # every combination of the four bits
    traj["n_deficit"][5] = 30  # 26 x (30 + 20) slots: the record runs past the capacity and is cut
    traj["n_additional"][5] = 20
    res["flags"][5] |= _abi.FLAG_RECORD_OVERFLOW
    got, d_acc = _accumulate(gpu_ctx, res, traj, yearly, 1000)
    ref = eval_ref.reference_record(res, traj, yearly, first_global=1000)
    assert eval_ref.counter_bytes(got) == eval_ref.counter_bytes(ref)
    hist = got.view("score_hist")
    assert hist[0] >= 1 and hist[2047] >= 2 and hist[1] >= 1 and got.score_out_of_range == 3
    assert got.view("flag_counts").tolist() == [int(((res["flags"] >> b) & 1).sum()) for b in range(4)]
    s = res["score"]
    assert (got.best_episode, got.worst_episode) == (1000 + int(np.nanargmax(s)), 1000 + int(np.nanargmin(s)))
    sm = got.view("final_metrics")[0]
    assert np.isnan(sm[0]) and sm[2] == np.nanmin(s) and sm[3] == np.nanmax(s)
    g, e = got.view("final_metrics")[1:], ref.view("final_metrics")[1:]
    assert np.array_equal(g[:, 2:], e[:, 2:])
    scale = np.maximum(np.abs(e[:, 2]), np.abs(e[:, 3]))
    np.testing.assert_array_less(np.abs(g[:, 0] - e[:, 0]), 1e-12 * np.abs(e[:, 0]) + 1e-13 * scale + 1e-300)
    # a second call accumulates: the record of both
    got2, _ = _accumulate(gpu_ctx, res[:100], traj[:100], yearly[:100], 1700, d_acc)
    assert got2.n_episodes == 800
    assert eval_ref.counter_bytes(got2) == eval_ref.counter_bytes(
        eval_ref.reference_record(np.concatenate([res, res[:100]]), np.concatenate([traj, traj[:100]]), np.concatenate([yearly, yearly[:100]])))


def test_edge_cases(gpu_ctx, trained):
    assert bytes(gpu_ctx.evaluate(trained, 0)) == bytes(_abi.EvalStats())
    one = gpu_ctx.evaluate(trained, 1, first_episode=77)
    assert one.n_episodes == 1 and one.best_episode == one.worst_episode == 77
    assert not one.view("final_metrics")[:, 1].any() and not one.view("yearly")[:, :, 1].any()
    res = gpu_ctx.rollout(trained, 1, first_episode=77)[0]
    assert one.view("final_metrics")[0, 0] == res["score"][0]


def test_errors(gpu_ctx, trained):
    L = _lib.lib()
    fresh = _lib.Context(0)
    with pytest.raises(_lib.EirgridError) as e:
        fresh.evaluate(trained, 10)
    assert e.value.code == -5
    fresh.close()
    with pytest.raises(_lib.EirgridError) as e:
        gpu_ctx.evaluate(trained, 10, cfg=_abi.RunCfg(enable_construction_delays=1))
    assert e.value.code == -1
    st = _abi.EvalStats()
    cfg = _abi.RunCfg()
    assert L.eg_evaluate(gpu_ctx.h, None, C.byref(cfg), 1, 0, 10, 1, C.byref(st)) == -1
    assert L.eg_evaluate(gpu_ctx.h, trained.h, None, 1, 0, 10, 1, C.byref(st)) == -1
    assert L.eg_evaluate(gpu_ctx.h, trained.h, C.byref(cfg), 1, 0, 10, 1, None) == -1
    assert L.eg_evaluate(None, trained.h, C.byref(cfg), 1, 0, 10, 1, C.byref(st)) == -1
    assert L.eg_eval_accumulate_device(gpu_ctx.h, None, None, None, 10, 0, None) == -1
    assert L.eg_eval_stats_merge(None, C.byref(st)) == -1 and L.eg_eval_stats_write_json(None, b"x.json") == -1


def test_synthetic_map():
    ctx = _lib.Context(0)
    ctx.map_set(*synthetic.scaled_map(ASSETS, factor=2))
    w = _lib.Weights()
    res, traj, _, yearly = ctx.rollout(w, 3000, seed=2, first_episode=11, want_yearly=True)
    got = ctx.evaluate(w, 3000, seed=2, first_episode=11)
    eval_ref.assert_record_matches(got, eval_ref.reference_record(res, traj, yearly, first_global=11), yearly=True)
    ctx.close()


def _env():
    return dict(os.environ, PYTHONPATH=ROOT)


def test_command_lines_write_the_record_of_the_call(gpu_ctx, trained, tmp_path):
    wpath = str(tmp_path / "w.json")
    trained.save_to_file(wpath)
    w = _lib.Weights.load_from_file(wpath)
    want = str(tmp_path / "want.json")
    gpu_ctx.evaluate(w, 5000, seed=4, first_episode=9, cfg=_abi.RunCfg(cost_only=1)).write_json(want)
    args = ["--weights", wpath, "--assets", ASSETS, "-n", "5000", "--seed", "4", "--first-episode", "9", "--cost-only"]
    py = str(tmp_path / "py.json")
    r = subprocess.run([sys.executable, "-m", "eirgrid_b200.evaluate"] + args + ["--json", py], capture_output=True, text=True, env=_env())
    assert r.returncode == 0, r.stderr
    subprocess.run(["make", "-C", os.path.join(ROOT, "host")], capture_output=True, check=True)
    host = str(tmp_path / "host.json")
    tool = os.path.join(ROOT, "host", "_build", "evaluate_policy")
    r = subprocess.run([tool] + args + ["--json", host, "--devices", "0"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert open(py, "rb").read() == open(want, "rb").read() == open(host, "rb").read()
    assert json.load(open(want))["episodes"] == 5000


def test_two_devices_agree(trained, tmp_path):
    torch = _torch()
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    wpath = str(tmp_path / "w.json")
    trained.save_to_file(wpath)
    args = ["--weights", wpath, "--assets", ASSETS, "-n", "70001", "--seed", "6"]
    tool = os.path.join(ROOT, "host", "_build", "evaluate_policy")
    subprocess.run(["make", "-C", os.path.join(ROOT, "host")], capture_output=True, check=True)
    out = {}
    for name, cmd in (("host1", [tool] + args + ["--devices", "0"]), ("host2", [tool] + args + ["--devices", "0,1"]),
                      ("torchrun2", [sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "-m", "eirgrid_b200.evaluate"] + args)):
        path = str(tmp_path / (name + ".json"))
        r = subprocess.run(cmd + ["--json", path], capture_output=True, text=True, env=_env())
        assert r.returncode == 0, (name, r.stderr[-2000:])
        out[name] = open(path, "rb").read()
    assert out["host2"] == out["torchrun2"]
    a, b = json.loads(out["host1"]), json.loads(out["host2"])
    for key in ("episodes", "flagged", "score_histogram", "best_episode", "worst_episode", "first_net_zero_year", "actions", "score_quantiles"):
        assert a[key] == b[key], key
    for f, m in a["final"].items():
        assert m["min"] == b["final"][f]["min"] and m["max"] == b["final"][f]["max"]
        assert m["mean"] == pytest.approx(b["final"][f]["mean"], rel=1e-12, abs=1e-12)
