"""numpy reference of the evaluation record (eg_eval_stats, csrc/evaluate.cu) built from episode arrays, and the comparison
the tests apply: integer parts, min/max and ids exact, means within 1e-12 and sums of squared deviations within 1e-10 relative
(with an absolute term scaled by the field's largest magnitude, see assert_record_matches)."""
import numpy as np

from eirgrid_b200 import _abi

N_Y, N_A, CAP = _abi.N_YEARS, _abi.N_ACTIONS, _abi.TRAJ_CAPACITY


def _moments(x):
    """rows of (mean, m2, min, max) over axis 0 of x [n, k]. The sums run in extended precision: numpy adds along axis 0
    one row after another, whose error (n eps of the values) would exceed that of the kernels' pairwise merges."""
    x = np.asarray(x, np.float64)
    out = np.zeros((x.shape[1], 4))
    for lo in range(0, x.shape[1], 32):
        c = x[:, lo:lo + 32].astype(np.longdouble)
        mean = c.mean(axis=0)
        out[lo:lo + 32, 0] = mean
        out[lo:lo + 32, 1] = ((c - mean) ** 2).sum(axis=0)
    out[:, 2], out[:, 3] = x.min(axis=0), x.max(axis=0)
    return out


def action_counts(traj):
    """(additional [26, 61], deficit [26, 61]) counted from the records as stored: rows cut at the capacity like the kernels"""
    nd = traj["n_deficit"].astype(np.int64)
    nrun = nd + traj["n_additional"].astype(np.int64)
    start = np.minimum(np.concatenate([np.zeros((len(traj), 1), np.int64), np.cumsum(nrun, axis=1)[:, :-1]], axis=1), CAP)
    nrun = np.minimum(nrun, CAP - start)
    nd = np.minimum(nd, nrun)
    add = np.zeros(N_Y * N_A, np.int64)
    dfc = np.zeros(N_Y * N_A, np.int64)
    s = np.arange(CAP)
    for lo in range(0, len(traj), 1024):
        st, nr, dd = start[lo:lo + 1024, :, None], nrun[lo:lo + 1024, :, None], nd[lo:lo + 1024, :, None]
        act = traj["actions"][lo:lo + 1024].astype(np.int64)
        inrow = (s >= st) & (s < st + nr)
        pos = s - st
        for mask, out in ((inrow & (pos < dd), dfc), (inrow & (pos >= dd), add)):
            e, y, slot = np.nonzero(mask)
            a = act[e, slot]
            ok = a < N_A
            out += np.bincount(y[ok] * N_A + a[ok], minlength=N_Y * N_A)
    return add.reshape(N_Y, N_A), dfc.reshape(N_Y, N_A)


def reference_record(res, traj, yearly=None, first_global=0):
    """eg_eval_stats of the episodes (res, traj, yearly) with global ids first_global.. (finite scores)"""
    st = _abi.EvalStats()
    n = len(res)
    st.n_episodes = n
    if n == 0:
        return st
    score = res["score"]
    st.best_episode = first_global + int(np.argmax(score))
    st.worst_episode = first_global + int(np.argmin(score))
    st.view("final_metrics")[:] = _moments(np.stack([res[f].astype(np.float64) for f in _abi.FINAL_FIELDS], axis=1))
    flags = res["flags"].astype(np.int64)
    st.n_flagged = int((flags != 0).sum())
    st.view("flag_counts")[:] = [int(((flags >> b) & 1).sum()) for b in range(_abi.EVAL_N_FLAGS)]
    inr = (score >= 0.0) & (score <= 2.0)
    st.view("score_hist")[:] = np.bincount(np.minimum(np.floor(score[inr] * 1024.0).astype(np.int64), _abi.EVAL_SCORE_BINS - 1),
                                           minlength=_abi.EVAL_SCORE_BINS)
    st.score_out_of_range = int((~inr).sum())
    add, dfc = action_counts(traj)
    st.view("additional_actions")[:] = add
    st.view("deficit_actions")[:] = dfc
    if yearly is not None:
        st.has_yearly = 1
        y = yearly["y"]
        vals = np.stack([y[f].astype(np.float64) for f in _abi.EVAL_YEAR_FIELDS], axis=2)  # [n, 26, 18]
        st.view("yearly")[:] = _moments(vals.reshape(n, -1)).reshape(N_Y, len(_abi.EVAL_YEAR_FIELDS), 4)
        nz = y["net_co2_emissions"] <= 0.0
        st.view("net_zero_or_below")[:] = nz.sum(axis=0)
        st.view("in_deficit")[:] = (y["power_balance"] < 0.0).sum(axis=0)
        first = np.where(nz.any(axis=1), np.argmax(nz, axis=1), N_Y)
        st.view("first_net_zero_year")[:] = np.bincount(first, minlength=N_Y + 1)
    return st


COUNTERS = ["n_flagged", "flag_counts", "score_hist", "score_out_of_range", "net_zero_or_below", "in_deficit", "first_net_zero_year",
            "additional_actions", "deficit_actions"]


def counter_bytes(st):
    return bytes(st)[_abi.EvalStats.n_flagged.offset:]


def assert_record_matches(got, exp, yearly=True):
    """integer parts, min/max and ids exact; moments within the tolerances below"""
    assert (got.n_episodes, got.has_yearly) == (exp.n_episodes, exp.has_yearly)
    assert (got.best_episode, got.worst_episode) == (exp.best_episode, exp.worst_episode)
    for name in COUNTERS:
        np.testing.assert_array_equal(got.view(name), exp.view(name), err_msg=name)
    parts = ["final_metrics"] + (["yearly"] if yearly else [])
    for name in parts:
        g, e = got.view(name).reshape(-1, 4), exp.view(name).reshape(-1, 4)
        np.testing.assert_array_equal(g[:, 2:], e[:, 2:], err_msg=name + " min/max")
        # plus a term relative to the field's largest magnitude: where values of both signs cancel, the mean is small against
        # the values and the rounding of any summation order is relative to the values
        scale = np.maximum(np.abs(e[:, 2]), np.abs(e[:, 3]))
        np.testing.assert_array_less(np.abs(g[:, 0] - e[:, 0]), 1e-12 * np.abs(e[:, 0]) + 1e-13 * scale + 1e-300, err_msg=name + " mean")
        n = max(int(exp.n_episodes), 1)
        np.testing.assert_array_less(np.abs(g[:, 1] - e[:, 1]), 1e-10 * np.abs(e[:, 1]) + 1e-12 * n * scale ** 2 + 1e-300,
                                     err_msg=name + " m2")
