"""The native (C++) host driver host/eirgrid_host.cpp: builds against the C ABI only, fails loudly without a GPU, and on a
GPU runs the batch/checkpoint loop with the reference's run-directory layout and resume rule."""
import json
import os
import subprocess

import pytest

from eirgrid_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ASSETS = os.path.join(ROOT, "tests", "golden", "ireland_map")
HOST = os.path.join(ROOT, "host", "_build", "eirgrid_host")


@pytest.fixture(scope="module")
def host_binary():
    from eirgrid_b200 import build
    build.build()
    r = subprocess.run(["make", "-C", os.path.join(ROOT, "host")], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    return HOST


def test_host_links_only_the_c_abi(host_binary):
    out = subprocess.run(["ldd", host_binary], capture_output=True, text=True).stdout
    assert "libeirgrid_b200.so" in out
    src = open(os.path.join(ROOT, "host", "eirgrid_host.cpp")).read()
    assert "cuda_runtime" not in src and "oracle" not in src.replace("// ", "")
    help_text = subprocess.run([host_binary, "--help"], capture_output=True, text=True).stdout
    for flag in ("--iterations", "--no-continue", "--checkpoint-dir", "--checkpoint-interval", "--progress-interval", "--cache-dir",
                 "--force-full-simulation", "--seed", "--cost-only", "--enable-energy-sales", "--enable-construction-delays",
                 "--track-weight-history"):
        assert flag in help_text, flag


def test_host_fails_loudly_without_gpu(host_binary):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = subprocess.run([host_binary, "-n", "10", "--assets", ASSETS, "--no-continue"], capture_output=True, text=True)
    assert r.returncode != 0 and "no CUDA device" in r.stderr and "no CPU fallback" in r.stderr


def test_host_rejects_malformed_arguments(host_binary):
    """Like clap on the reference's Args (cli/cli.rs:4-62): a usage error, never an abort or a wrapped-around number."""
    for args in (["-n", "abc"], ["-n", "-5"], ["-n", "99999999999999999999"], ["--devices", "x"], ["--batch-size", "5000000000"],
                 ["--batch-size", "0"], ["--update-mode", "weird"], ["--update-mode", "sequential-host"], ["--seed", "1.5"], ["--nonexistent"], ["-n"]):
        r = subprocess.run([host_binary] + args, capture_output=True, text=True)
        assert r.returncode == 2 and r.stderr.startswith("error: "), (args, r.returncode, r.stderr[:200])
        assert "terminate called" not in r.stderr


@pytest.mark.gpu
def test_host_run_checkpoint_and_resume(host_binary, tmp_path):
    ck = str(tmp_path / "ck")
    cache = str(tmp_path / "cache")
    os.makedirs(cache)
    open(os.path.join(cache, "location_analysis.json"), "w").write("{}")
    cmd = [host_binary, "--assets", ASSETS, "-c", ck, "-C", cache, "--batch-size", "2048", "--master-seed", "7", "-i", "1000"]
    r = subprocess.run(cmd + ["-n", "8192", "--no-continue"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    s1 = json.loads(r.stdout.strip().split("\n")[-1])
    assert s1["iterations"] == 8192 and s1["best_score"] is not None and s1["kernel_launches"] > 0
    run1 = s1["run_dir"]
    assert os.path.basename(run1).startswith("2024") and len(os.path.basename(run1)) == 15
    for f in ("latest_weights.json", "best_weights.json", "checkpoint_iteration.txt"):
        assert os.path.exists(os.path.join(run1, f)), f
    assert open(os.path.join(run1, "checkpoint_iteration.txt")).read().strip() == "8192"
    w = _lib.Weights.load_from_file(os.path.join(run1, "latest_weights.json"))
    assert w.table().iteration_count == 8192 and w.has_best_actions()
    # resume: continues from iteration 8192 with the saved weights; the last 10 % replay the best strategy
    import time
    time.sleep(1.1)  # a new timestamp directory
    r = subprocess.run(cmd + ["-n", "12288"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    s2 = json.loads(r.stdout.strip().split("\n")[-1])
    assert s2["start_iteration"] == 8192 and s2["iterations"] == 12288 and s2["run_dir"] != run1
    # an iteration count that is no multiple of the batch size is honoured exactly (the last batches are smaller)
    r = subprocess.run(cmd + ["-n", "5000", "--no-continue", "-c", str(tmp_path / "ck2")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    s3 = json.loads(r.stdout.strip().split("\n")[-1])
    assert s3["iterations"] == 5000 and s3["training_batches"]["episodes"] == 4500
    assert s2["best_score"] >= s1["best_score"]


@pytest.mark.gpu
def test_host_equals_python_driver(host_binary, tmp_path):
    """Same arguments, same seed: the C++ driver and the Python driver (run_multi_simulation) end with bit-identical weights —
    training batches through the device statistics path (eg_train_batch_* + eg_update_combine_apply vs the torch plumbing),
    a shorter last training batch, then the replay phase through the sequential update."""
    import numpy as np
    from eirgrid_b200.simulation import run_multi_simulation
    cache = str(tmp_path / "cache")
    os.makedirs(cache)
    open(os.path.join(cache, "location_analysis.json"), "w").write("{}")
    # 8192 iterations, batch 4096: training batches of 4096 and 3277 (up to iteration 7373), then 819 replay iterations
    r = subprocess.run([host_binary, "--assets", ASSETS, "-c", str(tmp_path / "ck_host"), "-C", cache, "--batch-size", "4096",
                        "--master-seed", "11", "-n", "8192", "--no-continue", "-i", "100000"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    s = json.loads(r.stdout.strip().split("\n")[-1])
    assert s["iterations"] == 8192 and s["training_batches"]["episodes"] == 7373
    py = run_multi_simulation(ASSETS, 8192, continue_from_checkpoint=False, checkpoint_dir=str(tmp_path / "ck_py"), checkpoint_interval=100000,
                              cache_dir=cache, batch_size=4096, master_seed=11, device=0, log=lambda *a: None)
    assert py["iterations"] == 8192
    got = _lib.Weights.load_from_file(os.path.join(s["run_dir"], "latest_weights.json"))
    want = _lib.Weights.load_from_file(os.path.join(py["run_dir"], "latest_weights.json"))
    tg, tw = got.table(), want.table()
    assert tg.iteration_count == tw.iteration_count == 8192
    assert tg.iterations_without_improvement == tw.iterations_without_improvement
    assert np.array_equal(np.ctypeslib.as_array(tg.weights), np.ctypeslib.as_array(tw.weights))
    assert np.array_equal(np.ctypeslib.as_array(tg.deficit_weights), np.ctypeslib.as_array(tw.deficit_weights))
    assert list(tg.best_metrics) == list(tw.best_metrics)
    bg, bw = got.best(), want.best()
    assert all(np.array_equal(x, y) for x, y in zip(bg[1] + bg[2], bw[1] + bw[2]))


@pytest.mark.gpu
def test_host_two_gpus_equal_one_gpu(host_binary, tmp_path):
    """Sharding a batch over GPUs changes nothing: --devices 0,1 with half the per-GPU batch ends with the weights of one GPU."""
    import numpy as np
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cache = str(tmp_path / "cache")
    os.makedirs(cache)
    open(os.path.join(cache, "location_analysis.json"), "w").write("{}")
    out = []
    for devs, batch, ck in (("0", "4096", "ck1"), ("0,1", "2048", "ck2")):
        r = subprocess.run([host_binary, "--assets", ASSETS, "-c", str(tmp_path / ck), "-C", cache, "--batch-size", batch, "--master-seed", "3",
                            "-n", "16384", "--no-continue", "-i", "100000", "--devices", devs], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        s = json.loads(r.stdout.strip().split("\n")[-1])
        out.append(_lib.Weights.load_from_file(os.path.join(s["run_dir"], "latest_weights.json")).table())
    assert np.array_equal(np.ctypeslib.as_array(out[0].weights), np.ctypeslib.as_array(out[1].weights))
    assert np.array_equal(np.ctypeslib.as_array(out[0].deficit_weights), np.ctypeslib.as_array(out[1].deficit_weights))
    assert list(out[0].best_metrics) == list(out[1].best_metrics)


@pytest.mark.gpu
def test_host_two_gpus_export_best_run_csv(host_binary, tmp_path):
    """The CSV export replays the best run on the first GPU's context while the second GPU, which ran the last training batch,
    is still the current device: the replay must run on the first context's device and export what one GPU exports."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cache = str(tmp_path / "cache")
    os.makedirs(cache)
    open(os.path.join(cache, "location_analysis.json"), "w").write("{}")
    summaries = []
    for devs, ck in (("0", "ck1"), ("0,1", "ck2")):
        r = subprocess.run([host_binary, "--assets", ASSETS, "-c", str(tmp_path / ck), "-C", cache, "--master-seed", "5", "-n", "9",
                            "--no-continue", "--devices", devs], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        s = json.loads(r.stdout.strip().split("\n")[-1])
        assert s["training_batches"]["episodes"] == 9 and "Enhanced simulation results exported to" in r.stdout
        (export,) = os.listdir(os.path.join(s["run_dir"], "enhanced_csv"))
        out = os.path.join(s["run_dir"], "enhanced_csv", export)
        for f in ("yearly_details/settlements.csv", "yearly_details/generators.csv", "yearly_details/carbon_offsets.csv",
                  "operation_logs/generator_operation_logs.csv"):
            assert os.path.exists(os.path.join(out, f)), f
        summaries.append([l for l in open(os.path.join(out, "simulation_summary.csv")) if not l.startswith("Timestamp,")])
    assert summaries[0] == summaries[1]


def test_analyze_locations_tool_flags_and_failure_without_gpu(host_binary):
    """host/analyze_locations.cpp mirrors aiSimulator/bin/analyze_locations.rs:7-17 (flags -m / -o / -c with the same defaults)"""
    tool = os.path.join(os.path.dirname(host_binary), "analyze_locations")
    assert os.path.exists(tool)
    out = subprocess.run([tool, "--help"], capture_output=True, text=True)
    assert out.returncode == 0
    for flag in ("--min-suitability", "--output-file", "--cache-dir", "0.3", "location_analysis.txt", "cache"):
        assert flag in out.stdout
    bad = subprocess.run([tool, "--min-suitability", "abc"], capture_output=True, text=True)
    assert bad.returncode == 2 and "invalid value" in bad.stderr
    import torch
    if not torch.cuda.is_available():
        r = subprocess.run([tool, "--assets", ASSETS], capture_output=True, text=True)
        assert r.returncode == 2 and "no CPU fallback" in r.stderr


@pytest.mark.gpu
def test_analyze_locations_tool_writes_both_files(host_binary, tmp_path):
    tool = os.path.join(os.path.dirname(host_binary), "analyze_locations")
    cache, txt = str(tmp_path / "cache"), str(tmp_path / "location_analysis.txt")
    # (0.2: the shipped cache holds scores down to 0.24, so it was written with a threshold below the tool's default of 0.3)
    r = subprocess.run([tool, "--assets", ASSETS, "-c", cache, "-o", txt, "-m", "0.2"], capture_output=True, text=True)
    assert r.returncode == 0 and "Analysis complete!" in r.stdout, r.stderr
    d = json.load(open(os.path.join(cache, "location_analysis.json")))
    assert len(d["locations"]) == 2601 and d["type_counts"]["OnshoreWind"] == 2601 and d["type_counts"]["OffshoreWind"] == 2421
    assert open(txt).read().startswith("Location Analysis Results\n========================\n\nTotal suitable locations: 2601\n")
