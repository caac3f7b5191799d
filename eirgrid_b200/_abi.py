"""Binary layouts of include/eirgrid_b200.h as numpy structured dtypes and ctypes structures.

Only layouts live here (no compute); both the product binding (eirgrid_b200/_lib.py) and the
test-side oracle loader (tests/oracle_lib.py) use them so that buffers can be compared field by field.
"""
import ctypes as C

import numpy as np

BASE_YEAR = 2025
END_YEAR = 2050
N_YEARS = 26
N_GEN_TYPES = 15
N_ACTIONS = 61
N_DEFICIT_KEYS = 15
N_COUNT_KEYS = 21
TRAJ_CAPACITY = 984   # action slots per episode record (EG_TRAJ_CAPACITY); year rows are stored back to back
BEST_CAPACITY = 2 * TRAJ_CAPACITY
SITE_NONE = 0xFFFF
ACT_DO_NOTHING = 60

FLAG_GEN_OVERFLOW = 1
FLAG_OFFSET_OVERFLOW = 2
FLAG_RECORD_OVERFLOW = 4
FLAG_NO_SITE = 8

GEN_TYPES = ["OnshoreWind", "OffshoreWind", "DomesticSolar", "CommercialSolar", "UtilitySolar", "Nuclear",
             "CoalPlant", "GasCombinedCycle", "GasPeaker", "Biomass", "HydroDam", "PumpedStorage",
             "BatteryStorage", "TidalGenerator", "WaveEnergy"]  # models/generator.rs:11-36
OFFSET_TYPES = ["Forest", "Wetland", "ActiveCapture", "CarbonCredit"]  # weights/core.rs:100-114 insertion order
MULTS = [100, 120, 150]

RESULT_DTYPE = np.dtype([
    ("score", "<f8"), ("net_emissions", "<f8"), ("public_opinion", "<f8"), ("total_cost", "<f8"),
    ("power_reliability", "<f8"), ("n_generators", "<u4"), ("n_offsets", "<u4"),
    ("n_deficit_actions", "<u2"), ("n_additional_actions", "<u2"), ("flags", "<u4"), ("reserved", "<u4"),
    ("_pad", "<u4")], align=False)
assert RESULT_DTYPE.itemsize == 64

TRAJ_DTYPE = np.dtype([
    ("n_deficit", "<u2", (N_YEARS,)), ("n_additional", "<u2", (N_YEARS,)),
    ("actions", "u1", (TRAJ_CAPACITY,))])
assert TRAJ_DTYPE.itemsize == 1088

SITES_DTYPE = np.dtype([("site", "<u2", (TRAJ_CAPACITY,))])
assert SITES_DTYPE.itemsize == 1968


def traj_row_starts(traj):
    """First slot of each year's row: int array [..., 27] (last entry = slots used) for one record or an array of records."""
    n = traj["n_deficit"].astype(np.int64) + traj["n_additional"].astype(np.int64)
    return np.concatenate([np.zeros(n.shape[:-1] + (1,), np.int64), np.cumsum(n, axis=-1)], axis=-1)


def traj_rows(rec, values=None):
    """The 26 year rows of ONE record as a list of (deficit part, additional part) arrays; `values` = the per-slot
    array to slice (default: the record's actions; pass sites["site"] for the placement sites)."""
    a = rec["actions"] if values is None else values
    start = traj_row_starts(rec)
    out = []
    for y in range(N_YEARS):
        nd = int(rec["n_deficit"][y])
        out.append((a[start[y]:start[y] + nd], a[start[y] + nd:start[y + 1]]))
    return out


def pack_traj(rows):
    """Inverse of traj_rows: rows = 26 x (deficit actions, additional actions) -> one TRAJ_DTYPE record."""
    rec = np.zeros((), TRAJ_DTYPE)
    pos = 0
    for y, (d, a) in enumerate(rows):
        d, a = np.asarray(d, np.uint8), np.asarray(a, np.uint8)
        if pos + len(d) + len(a) > TRAJ_CAPACITY:
            raise ValueError("record exceeds TRAJ_CAPACITY")
        rec["n_deficit"][y], rec["n_additional"][y] = len(d), len(a)
        rec["actions"][pos:pos + len(d)] = d
        rec["actions"][pos + len(d):pos + len(d) + len(a)] = a
        pos += len(d) + len(a)
    return rec

YEAR_FIELDS = ["total_power_usage", "total_power_generation", "power_balance", "average_public_opinion",
               "yearly_capital_cost", "total_capital_cost", "inflation_factor", "total_co2_emissions",
               "total_carbon_offset", "net_co2_emissions", "yearly_carbon_credit_revenue",
               "total_carbon_credit_revenue", "yearly_energy_sales_revenue", "total_energy_sales_revenue",
               "yearly_total_cost", "total_cost", "reserved"]
YEAR_DTYPE = np.dtype([("total_population", "<u4"), ("active_generators", "<u4")] + [(f, "<f8") for f in YEAR_FIELDS])
assert YEAR_DTYPE.itemsize == 144
YEARLY_DTYPE = np.dtype([("y", YEAR_DTYPE, (N_YEARS,))])

STATS_WORDS = 8 + N_YEARS * (3 * N_ACTIONS + N_DEFICIT_KEYS)


class RunCfg(C.Structure):
    _fields_ = [("cost_only", C.c_uint32), ("enable_energy_sales", C.c_uint32),
                ("enable_construction_delays", C.c_uint32), ("replay_best", C.c_uint32),
                ("same_stream_all_episodes", C.c_uint32), ("reserved", C.c_uint32 * 3)]

    def __init__(self, cost_only=0, enable_energy_sales=1, enable_construction_delays=0, replay_best=0,
                 same_stream_all_episodes=0):
        super().__init__(int(cost_only), int(enable_energy_sales), int(enable_construction_delays),
                         int(replay_best), int(same_stream_all_episodes))


class MapDesc(C.Structure):
    _fields_ = [("n_settlements", C.c_uint32), ("settlement_x", C.POINTER(C.c_double)),
                ("settlement_y", C.POINTER(C.c_double)), ("settlement_pop", C.POINTER(C.c_uint32)),
                ("n_existing", C.c_uint32), ("existing_x", C.POINTER(C.c_double)),
                ("existing_y", C.POINTER(C.c_double)), ("existing_type", C.POINTER(C.c_uint8)),
                ("existing_capacity_mw", C.POINTER(C.c_double)),
                ("n_coast", C.c_uint32), ("coast_x", C.POINTER(C.c_double)), ("coast_y", C.POINTER(C.c_double)),
                ("grid_n", C.c_uint32), ("grid_step", C.c_double)]


class WeightsTable(C.Structure):
    _fields_ = [("weights", (C.c_double * N_ACTIONS) * N_YEARS),
                ("deficit_weights", (C.c_double * N_DEFICIT_KEYS) * N_YEARS),
                ("count_weights", (C.c_double * N_COUNT_KEYS) * N_YEARS),
                ("learning_rate", C.c_double), ("exploration_rate", C.c_double),
                ("best_metrics", C.c_double * 4),
                ("has_count_weights", C.c_uint32), ("has_best", C.c_uint32),
                ("iteration_count", C.c_uint32), ("iterations_without_improvement", C.c_uint32)]

    def arrays(self):
        """(weights[26,61], deficit[26,15], count[26,21]) as numpy copies."""
        return (np.ctypeslib.as_array(self.weights).copy(), np.ctypeslib.as_array(self.deficit_weights).copy(),
                np.ctypeslib.as_array(self.count_weights).copy())


class UpdateStats(C.Structure):
    _fields_ = [("n_episodes", C.c_uint32), ("n_improvements", C.c_uint32), ("n_contrast_applied", C.c_uint32),
                ("iterations_without_improvement", C.c_uint32), ("best_score", C.c_double),
                ("batch_best_score", C.c_double), ("batch_best_episode", C.c_int64), ("n_flagged", C.c_uint32), ("reserved", C.c_uint32)]


EVAL_CHUNK = 65536
EVAL_SCORE_BINS = 2048
EVAL_N_FLAGS = 4
FINAL_FIELDS = ["score", "net_emissions", "public_opinion", "total_cost", "power_reliability", "n_generators", "n_offsets",
                "n_deficit_actions", "n_additional_actions"]
EVAL_YEAR_FIELDS = ["total_population", "active_generators"] + YEAR_FIELDS[:-1]  # every field of eg_year_metrics but `reserved`
MOMENTS = ["mean", "m2", "min", "max"]


class EvalStats(C.Structure):
    """eg_eval_stats: statistics of an evaluation (Context.evaluate). Moment arrays are [..., 4] = (mean, m2, min, max); the
    numpy views share the structure's memory. The all-zero structure is the empty statistics."""
    _fields_ = [("n_episodes", C.c_uint64), ("best_episode", C.c_uint64), ("worst_episode", C.c_uint64),
                ("has_yearly", C.c_uint32), ("reserved", C.c_uint32),
                ("final_metrics", (C.c_double * 4) * len(FINAL_FIELDS)),
                ("yearly", ((C.c_double * 4) * len(EVAL_YEAR_FIELDS)) * N_YEARS),
                ("n_flagged", C.c_uint64), ("flag_counts", C.c_uint64 * EVAL_N_FLAGS),
                ("score_hist", C.c_uint64 * EVAL_SCORE_BINS), ("score_out_of_range", C.c_uint64),
                ("net_zero_or_below", C.c_uint64 * N_YEARS), ("in_deficit", C.c_uint64 * N_YEARS),
                ("first_net_zero_year", C.c_uint64 * (N_YEARS + 1)),
                ("additional_actions", (C.c_uint64 * N_ACTIONS) * N_YEARS), ("deficit_actions", (C.c_uint64 * N_ACTIONS) * N_YEARS)]

    def view(self, name):
        """numpy view of an array field (e.g. view("final_metrics")[FINAL_FIELDS.index("score"), 0] is the mean score)"""
        return np.ctypeslib.as_array(getattr(self, name))

    def moments(self, field, year=None):
        """{mean, m2, min, max} of a final metric, or of a yearly field in year index `year`"""
        row = self.view("final_metrics")[FINAL_FIELDS.index(field)] if year is None else \
            self.view("yearly")[year, EVAL_YEAR_FIELDS.index(field)]
        return dict(zip(MOMENTS, (float(v) for v in row)))

    def merge(self, other):
        """self <- self followed by other (eg_eval_stats_merge); returns self"""
        from . import _lib
        _lib.check(_lib.lib().eg_eval_stats_merge(C.byref(self), C.byref(other)))
        return self

    def write_json(self, path):
        """the record as JSON (eg_eval_stats_write_json)"""
        import os
        from . import _lib
        _lib.check(_lib.lib().eg_eval_stats_write_json(C.byref(self), os.fsencode(path)))

    @classmethod
    def from_bytes(cls, data):
        return cls.from_buffer_copy(bytes(data))


def action_name(code):
    """Human-readable GridAction for an action code (ai/actions/grid_action.rs:18-40 Display format)."""
    if code < 45:
        return "AddGenerator(%s, %d%%)" % (GEN_TYPES[code // 3], MULTS[code % 3])
    if code < 57:
        return "AddCarbonOffset(%s, %d%%)" % (OFFSET_TYPES[(code - 45) // 3], MULTS[(code - 45) % 3])
    return {57: "UpgradeEfficiency()", 58: "AdjustOperation(, 0%)", 59: "CloseGenerator()", 60: "DoNothing"}[code]


def ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None
