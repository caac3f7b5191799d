"""numpy restatement of the batch-synchronous update statistics (DESIGN.md §update), used to check
eirgrid_b200/csrc/stats.cu and to drive the CPU (gloo) test of the multi-rank combine step."""
import math

import numpy as np

from eirgrid_b200 import _abi

HEADER = 8
YEAR_STRIDE = 3 * _abi.N_ACTIONS + _abi.N_DEFICIT_KEYS
FIXED = 16777216.0
DEFICIT_KEY_TYPE = [8, 7, 12, 11, 9, 0, 1, 4, 10, 5, 2, 3, 13, 14]


def default_score(net, opinion, cost, cost_only=False):
    normalized = max(cost / 50000000000.0, 1.0)
    if cost_only:
        return 2.0 - min(math.log(normalized) / math.log(100.0), 1.0)
    if net > 0.0:
        return 1.0 - min(net / 1000000.0, 1.0)
    cost_score = 1.0 - min(math.log(normalized) / math.log(100.0), 1.0)
    cw = 0.8 if normalized > 8.0 else 0.5
    return 1.0 + (cost_score * cw + opinion * (1.0 - cw))


def deficit_key(code):
    if code == 60:
        return 14
    if code < 45 and code % 3 == 0 and code // 3 in DEFICIT_KEY_TYPE:
        return DEFICIT_KEY_TYPE.index(code // 3)
    return -1


def contrast_consts(table, cost_only=False):
    """The constants of one batch, with the stored best metrics scored in the weights' optimisation mode."""
    iwi = table.iterations_without_improvement
    stag = 1.0 + 0.2 * (iwi / 10.0) ** 1.8
    alr = table.learning_rate * (1.0 + 0.1 * iwi)
    best_score = default_score(*list(table.best_metrics)[:3], cost_only=cost_only) if table.has_best else 0.0
    return dict(has_best=bool(table.has_best), force=iwi > 800, best_score=best_score, cost_only=cost_only,
                threshold=0.1 * max(math.exp(-iwi / 500.0), 0.00001 / 0.1), stagnation=stag, alr=alr)


def recorded_rows(t):
    """(run, deficit) action lists of each year as the update reads a record: year rows follow each other, and counts that
    run past the record's capacity are cut (eg_traj_next_row in csrc/traj_rows.hpp)."""
    rows, row = [], 0
    a = t["actions"]
    for y in range(_abi.N_YEARS):
        nd = min(int(t["n_deficit"][y]), _abi.TRAJ_CAPACITY - row)
        na = min(int(t["n_additional"][y]), _abi.TRAJ_CAPACITY - row - nd)
        rows.append(([int(x) for x in a[row:row + nd + na]], [int(x) for x in a[row:row + nd]]))
        row += nd + na
    return rows


def batch_stats(results, trajs, consts, best, best_deficit):
    """best / best_deficit: per-year lists of action codes of the snapshot's best strategy.
    Returns (statistics table, scores, terms): terms[w] is the number of values summed into word w."""
    stats = np.zeros(_abi.STATS_WORDS, np.int64)
    terms = np.zeros(_abi.STATS_WORDS, np.int64)
    scores = np.zeros(len(results))
    cbs = [list(best[y]) + list(best_deficit[y]) for y in range(_abi.N_YEARS)]
    for e in range(len(results)):
        r, t = results[e], trajs[e]
        score = default_score(float(r["net_emissions"]), float(r["public_opinion"]), float(r["total_cost"]), consts["cost_only"])
        scores[e] = score
        stats[0] += 1
        stats[2] += int(r["flags"] != 0)
        passed = False
        log_pen = log_mild = 0
        if consts["has_best"]:
            det = (consts["best_score"] - score) / consts["best_score"] if consts["best_score"] > 0 else 0.0
            passed = det > consts["threshold"] or consts["force"]
            if passed:
                if det < 0:
                    log_pen = log_mild = -(1 << 40)
                else:
                    combined = det ** 0.3 * consts["stagnation"]
                    log_pen = int(np.rint(math.log(1.0 / (1.0 + consts["alr"] * 1.5 * combined)) * FIXED))
                    log_mild = int(np.rint(math.log(1.0 / (1.0 + consts["alr"] * combined * 0.5)) * FIXED))
                stats[1] += 1
        for y, (run, deficit) in enumerate(recorded_rows(t)):
            base = HEADER + y * YEAR_STRIDE
            cb = cbs[y]
            for i, a in enumerate(run + deficit):
                if i < len(run):
                    w = base + 2 * 61 + a
                else:
                    k = deficit_key(a)
                    w = base + 3 * 61 + k if k >= 0 else -1
                if w >= 0:
                    stats[w] += 1
                    terms[w] += 1
                if not passed:
                    continue
                if a not in cb:
                    stats[base + a] += log_pen
                    terms[base + a] += 1
                elif i < len(cb) and cb[i] != a:
                    stats[base + 61 + a] += log_mild
                    terms[base + 61 + a] += 1
    return stats, scores, terms


def assert_stats_match(got, best_score, best_index, exp, scores, terms):
    """The statistics kernel's output against batch_stats: header words and occurrence counts exact; each fixed-point log
    word within its number of terms (device log()/pow() may differ from libm in the last bit, which moves one llrint by at
    most one unit); the same words non-zero; the best score within 1e-12 and the lowest index among equal best scores."""
    got = np.asarray(got, np.int64)
    assert np.array_equal(got[:HEADER], exp[:HEADER]), (got[:HEADER], exp[:HEADER])
    g = got[HEADER:].reshape(_abi.N_YEARS, YEAR_STRIDE)
    e = exp[HEADER:].reshape(_abi.N_YEARS, YEAR_STRIDE)
    k = terms[HEADER:].reshape(_abi.N_YEARS, YEAR_STRIDE)
    assert np.array_equal(g[:, 2 * _abi.N_ACTIONS:], e[:, 2 * _abi.N_ACTIONS:])
    d = np.abs(g[:, :2 * _abi.N_ACTIONS] - e[:, :2 * _abi.N_ACTIONS])
    assert (d <= k[:, :2 * _abi.N_ACTIONS]).all(), int((d - k[:, :2 * _abi.N_ACTIONS]).max())
    assert np.array_equal(g != 0, e != 0)
    if len(scores) == 0:
        assert best_score == -1.0 and best_index == (1 << 64) - 1
        return
    i = int(np.lexsort((np.arange(len(scores)), -scores))[0])
    assert best_index == i, (best_index, i)
    assert abs(best_score - scores[i]) <= 1e-12 * scores[i], (best_score, scores[i])
