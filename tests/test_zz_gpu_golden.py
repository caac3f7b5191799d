"""CUDA path against the COMMITTED golden vectors (tests/golden/oracle_frozen_r02.npz), without the oracle in the loop.

The fixture holds what the oracle produced when it was frozen (make_oracle_frozen.py); test_oracle.py checks on the CPU that
the oracle still produces it, this file checks that the GPU does. (Runs last: the file name sorts after the other suites.)
"""
import hashlib
import os

import numpy as np
import pytest

from eirgrid_b200 import _lib

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_frozen_r02.npz")
EXACT = ("net_emissions", "public_opinion", "total_cost", "power_reliability", "n_generators", "n_offsets", "n_deficit_actions",
         "n_additional_actions", "flags")


def _same_results(got, want):
    for f in EXACT:
        assert np.array_equal(got[f], want[f]), f
    np.testing.assert_allclose(got["score"], want["score"], rtol=1e-12, atol=0)  # ln evaluated on the device


def test_rollout_and_replay_equal_the_committed_vectors(gpu_ctx):
    g = np.load(GOLDEN)
    w = _lib.Weights()
    res, traj, sites, _ = gpu_ctx.rollout(w, 64, seed=1, first_episode=0, want_sites=True)
    assert traj.tobytes() == g["initial_traj"].tobytes()
    assert hashlib.sha1(sites.tobytes()).digest() == g["initial_sites_sha1"].tobytes()
    _same_results(res, g["initial_results"])
    # the lean (training) instantiation of the kernel: same episodes without the optional outputs
    res_l, traj_l, _, _ = gpu_ctx.rollout(w, 64, seed=1, first_episode=0)
    assert traj_l.tobytes() == g["initial_traj"].tobytes()
    _same_results(res_l, g["initial_results"])
    # 64 sequential reference-rule updates, then the three sampling regimes
    w.update(g["initial_results"], g["initial_traj"])
    t = w.table()
    assert hashlib.sha1(bytes(t)).digest() == g["updated_table_sha1"].tobytes()
    for iwi in (150, 600, 1300):
        t = w.table()
        t.iterations_without_improvement = iwi
        w.set_table(t)
        r2, t2, s2, _ = gpu_ctx.rollout(w, 32, seed=7 + iwi, first_episode=1000, want_sites=True)
        assert hashlib.sha1(t2.tobytes()).digest() == g["iwi%d_traj_sha1" % iwi].tobytes(), iwi
        assert hashlib.sha1(s2.tobytes()).digest() == g["iwi%d_sites_sha1" % iwi].tobytes(), iwi
        _same_results(r2, g["iwi%d_results" % iwi])
        if iwi > 500:  # the lean stagnation instantiation (no optional outputs): the same episodes
            r3, t3, _, _ = gpu_ctx.rollout(w, 32, seed=7 + iwi, first_episode=1000)
            assert hashlib.sha1(t3.tobytes()).digest() == g["iwi%d_traj_sha1" % iwi].tobytes(), iwi
            _same_results(r3, g["iwi%d_results" % iwi])
    rr, _, _ = gpu_ctx.replay(g["initial_traj"][:8])
    _same_results(rr, g["replay_results"])
