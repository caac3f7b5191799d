"""ctypes binding of libeirgrid_b200.so (the C ABI declared in include/eirgrid_b200.h).

The library is built in-tree by `python -m eirgrid_b200.build`. There is no Python or CPU fallback: if the
shared object is missing this module raises, and every compute call fails with EG_ERR_NO_DEVICE without a GPU.
"""
import ctypes as C
import os

import numpy as np

from . import _abi

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, os.environ.get("EIRGRID_LIB_NAME", "libeirgrid_b200.so"))  # side-by-side builds: A/B variants, -DEG_DEBUG_BOUNDS

EXPORTS = [
    "eg_init", "eg_destroy", "eg_last_error", "eg_sync", "eg_kernel_launches", "eg_map_load", "eg_map_set",
    "eg_map_info", "eg_map_site_tables", "eg_map_site_static", "eg_weights_new", "eg_weights_free",
    "eg_weights_clone", "eg_weights_load_json", "eg_weights_save_json", "eg_weights_merge", "eg_weights_get_table",
    "eg_weights_set_table", "eg_weights_get_best", "eg_deficit_key_action", "eg_rollout_batch", "eg_weights_upload",
    "eg_rollout_batch_device", "eg_replay_batch", "eg_replay_batch_device", "eg_update", "eg_update_stats_device",
    "eg_update_apply_stats", "eg_location_analysis", "eg_update_stats_clear_device", "eg_update_pack_best_device",
    "eg_location_analysis_year", "eg_microbench_fp64", "eg_export_best_run_csv", "eg_weights_history_append", "eg_train_batch_begin", "eg_train_batch_end", "eg_train_batch_results", "eg_update_combine_apply",
    "eg_update_device", "eg_train_batch_inorder", "eg_rule_math",
    "eg_location_analysis_sites", "eg_location_analysis_sites_device", "eg_location_analysis_write",
    "eg_update_pack_exchange_device",
]


class EirgridError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("eirgrid_b200 error %d: %s" % (code, message))
        self.code = code


_lib = None


def lib():
    """Load the CUDA library; raises if it has not been built (no silent fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("%s is missing: run `python -m eirgrid_b200.build` (needs nvcc). "
                          "eirgrid_b200 has no CPU fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, u32, u64, i64 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int64
    L.eg_last_error.restype = C.c_char_p
    L.eg_init.argtypes = [C.c_int, vp, C.POINTER(vp)]
    L.eg_destroy.argtypes = [vp]
    L.eg_destroy.restype = None
    L.eg_sync.argtypes = [vp]
    L.eg_kernel_launches.argtypes = [vp]
    L.eg_kernel_launches.restype = u64
    L.eg_map_load.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_char_p]
    L.eg_map_set.argtypes = [vp, C.POINTER(_abi.MapDesc)]
    L.eg_map_info.argtypes = [vp, C.POINTER(u32)]
    L.eg_map_site_tables.argtypes = [vp, u32, u32, u32, vp, vp, vp]
    L.eg_map_site_static.argtypes = [vp, vp, vp]
    L.eg_weights_new.argtypes = [C.POINTER(vp)]
    L.eg_weights_free.argtypes = [vp]
    L.eg_weights_free.restype = None
    L.eg_weights_clone.argtypes = [vp, C.POINTER(vp)]
    L.eg_weights_load_json.argtypes = [C.c_char_p, C.POINTER(vp)]
    L.eg_weights_save_json.argtypes = [vp, C.c_char_p]
    L.eg_weights_merge.argtypes = [vp, vp]
    L.eg_weights_get_table.argtypes = [vp, C.POINTER(_abi.WeightsTable)]
    L.eg_weights_set_table.argtypes = [vp, C.POINTER(_abi.WeightsTable)]
    L.eg_weights_get_best.argtypes = [vp, vp, vp, C.c_size_t, vp, vp, C.c_size_t]
    L.eg_deficit_key_action.argtypes = [u32]
    L.eg_deficit_key_action.restype = C.c_uint8
    L.eg_rollout_batch.argtypes = [vp, vp, C.POINTER(_abi.RunCfg), u64, u64, u32, vp, vp, vp, vp]
    L.eg_weights_upload.argtypes = [vp, vp]
    L.eg_rollout_batch_device.argtypes = [vp, C.POINTER(_abi.RunCfg), u64, u64, u32, vp, vp, vp, vp]
    L.eg_replay_batch.argtypes = [vp, C.POINTER(_abi.RunCfg), vp, u32, vp, vp, vp]
    L.eg_replay_batch_device.argtypes = [vp, C.POINTER(_abi.RunCfg), vp, u32, vp, vp, vp]
    L.eg_update.argtypes = [vp, vp, vp, u32, u32, u64, C.POINTER(_abi.UpdateStats)]
    L.eg_update_device.argtypes = [vp, vp, vp, vp, u32, u32, u64, C.POINTER(_abi.UpdateStats)]
    L.eg_train_batch_inorder.argtypes = [vp, vp, C.POINTER(_abi.RunCfg), u64, u64, u32, u64, C.POINTER(_abi.UpdateStats)]
    L.eg_update_stats_device.argtypes = [vp, vp, vp, vp, u32, vp, vp, vp]
    L.eg_update_stats_clear_device.argtypes = [vp, vp]
    L.eg_update_pack_exchange_device.argtypes = [vp, vp, vp, u32, vp, vp, vp, u64, vp, vp, u32, u32, u32, vp]
    L.eg_update_pack_best_device.argtypes = [vp, vp, vp, u32, vp, vp, u64, vp]
    L.eg_weights_history_append.argtypes = [vp, u64, C.c_char_p]
    L.eg_location_analysis_sites.argtypes = [vp, C.c_int, u32, C.c_double, u32, u32, u32, u32, vp]
    L.eg_location_analysis_sites_device.argtypes = [vp, C.c_int, u32, C.c_double, u32, u32, u32, u32, vp]
    L.eg_location_analysis_write.argtypes = [vp, C.c_int, C.c_double, C.c_char_p, C.c_char_p]
    L.eg_rule_math.argtypes = [C.c_int, u32, vp, vp, u32, vp]
    L.eg_microbench_fp64.argtypes = [C.c_int, C.POINTER(C.c_double)]
    L.eg_export_best_run_csv.argtypes = [vp, vp, C.POINTER(_abi.RunCfg), C.c_char_p, C.c_char_p]
    L.eg_train_batch_begin.argtypes = [vp, vp, C.POINTER(_abi.RunCfg), u64, u64, u32]
    L.eg_train_batch_end.argtypes = [vp, vp, vp]
    L.eg_train_batch_results.argtypes = [vp, vp, vp]
    L.eg_update_combine_apply.argtypes = [vp, vp, vp, u32, u64, u64, C.POINTER(_abi.UpdateStats)]
    L.eg_update_apply_stats.argtypes = [vp, vp, u64, vp, vp, i64, C.POINTER(_abi.UpdateStats)]
    L.eg_location_analysis.argtypes = [vp, C.c_int, C.c_int32, C.c_double, vp, u32, u32]
    L.eg_location_analysis_year.argtypes = [vp, C.c_int, u32, C.c_int32, C.c_double, vp, u32, u32]
    _lib = L
    return L


def check(rc):
    if rc < 0:
        raise EirgridError(rc, lib().eg_last_error().decode("utf-8", "replace"))
    return rc


def _dev_ptr(t):
    """Device pointer of a torch tensor (or None / int passthrough)."""
    if t is None:
        return None
    if isinstance(t, int):
        return t
    return t.data_ptr()


def rule_math(fn, x, y=None, device=-1):
    """Test aid: csrc/eg_math.hpp / csrc/update_rule.hpp evaluated on the host (device < 0) or on a GPU."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.zeros_like(x) if y is None else np.ascontiguousarray(np.broadcast_to(np.asarray(y, dtype=np.float64), x.shape))
    out = np.zeros_like(x)
    check(lib().eg_rule_math(int(device), int(fn), _abi.ptr(x), _abi.ptr(y), x.size, _abi.ptr(out)))
    return out


class Weights:
    """The policy table == reference ActionWeights (ai/learning/weights/mod.rs:49-107)."""

    def __init__(self, handle=None):
        self.L = lib()
        if handle is None:
            h = C.c_void_p()
            check(self.L.eg_weights_new(C.byref(h)))  # ActionWeights::new
            handle = h
        self.h = handle

    @classmethod
    def load_from_file(cls, path):  # ActionWeights::load_from_file
        h = C.c_void_p()
        check(lib().eg_weights_load_json(os.fsencode(path), C.byref(h)))
        return cls(h)

    def save_to_file(self, path):  # ActionWeights::save_to_file
        parent = os.path.dirname(path)
        if parent:
            os.makedirs(parent, exist_ok=True)
        check(self.L.eg_weights_save_json(self.h, os.fsencode(path)))

    def clone(self):
        h = C.c_void_p()
        check(self.L.eg_weights_clone(self.h, C.byref(h)))
        return Weights(h)

    def history_append(self, iteration, path):  # save_weight_history, multi_simulation.rs:179-207
        check(self.L.eg_weights_history_append(self.h, int(iteration), os.fsencode(path)))

    def update_weights_from(self, other):  # ActionWeights::update_weights_from
        check(self.L.eg_weights_merge(self.h, other.h))

    def table(self):
        t = _abi.WeightsTable()
        check(self.L.eg_weights_get_table(self.h, C.byref(t)))
        return t

    def set_table(self, t):
        check(self.L.eg_weights_set_table(self.h, C.byref(t)))

    def best(self):
        """(has_best, best_actions, best_deficit_actions): two lists of 26 uint8 arrays (any length, like the reference's Vecs)"""
        nb, nd = np.zeros(26, np.uint32), np.zeros(26, np.uint32)
        has = check(self.L.eg_weights_get_best(self.h, _abi.ptr(nb), None, 0, _abi.ptr(nd), None, 0))
        b, d = np.zeros(max(int(nb.sum()), 1), np.uint8), np.zeros(max(int(nd.sum()), 1), np.uint8)
        check(self.L.eg_weights_get_best(self.h, _abi.ptr(nb), _abi.ptr(b), b.size, _abi.ptr(nd), _abi.ptr(d), d.size))
        ob, od = np.concatenate([[0], np.cumsum(nb)]).astype(np.int64), np.concatenate([[0], np.cumsum(nd)]).astype(np.int64)
        return (bool(has), [b[ob[y]:ob[y + 1]].copy() for y in range(26)], [d[od[y]:od[y + 1]].copy() for y in range(26)])

    def has_best_actions(self):  # ActionWeights::has_best_actions
        return bool(self.table().has_best)

    def update(self, results, trajs, replay_best=False, rng_seed=0):
        """The write-lock section of multi_simulation.rs:494-508 for a batch, in episode order (host arrays)."""
        results = np.ascontiguousarray(results)
        trajs = np.ascontiguousarray(trajs)
        assert results.dtype == _abi.RESULT_DTYPE and trajs.dtype == _abi.TRAJ_DTYPE and len(results) == len(trajs)
        st = _abi.UpdateStats()
        check(self.L.eg_update(self.h, _abi.ptr(results), _abi.ptr(trajs), len(results), int(replay_best), rng_seed,
                               C.byref(st)))
        return st

    def apply_stats(self, stats, n_total, best_result, best_traj, best_index):
        stats = np.ascontiguousarray(stats, dtype=np.int64)
        assert stats.size == _abi.STATS_WORDS
        st = _abi.UpdateStats()
        br = np.ascontiguousarray(best_result) if best_result is not None else None
        bt = np.ascontiguousarray(best_traj) if best_traj is not None else None
        check(self.L.eg_update_apply_stats(self.h, _abi.ptr(stats), int(n_total), _abi.ptr(br), _abi.ptr(bt),
                                           int(best_index), C.byref(st)))
        return st

    def __del__(self):
        try:
            self.L.eg_weights_free(self.h)
        except Exception:
            pass


class Context:
    """One device context per process/GPU (eg_ctx)."""

    def __init__(self, device=0, stream=None):
        self.L = lib()
        h = C.c_void_p()
        check(self.L.eg_init(int(device), C.c_void_p(stream) if stream else None, C.byref(h)))
        self.h = h
        self.device = device

    def close(self):
        if self.h:
            self.L.eg_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- map ----
    def map_load(self, settlements_json, generators_csv, coastline_json):
        check(self.L.eg_map_load(self.h, os.fsencode(settlements_json), os.fsencode(generators_csv),
                                 os.fsencode(coastline_json)))

    def map_load_dir(self, asset_dir):
        """asset_dir holds settlements.json, ireland_generators.csv, coastline_points.json (aiSimulator/assets layout)."""
        self.map_load(os.path.join(asset_dir, "settlements.json"), os.path.join(asset_dir, "ireland_generators.csv"),
                      os.path.join(asset_dir, "coastline_points.json"))

    def map_set(self, sx, sy, spop, ex, ey, etype, ecap, cx, cy, grid_n, grid_step):
        f8 = lambda a: np.ascontiguousarray(a, dtype=np.float64)
        sx, sy, ex, ey, ecap, cx, cy = map(f8, (sx, sy, ex, ey, ecap, cx, cy))
        spop = np.ascontiguousarray(spop, dtype=np.uint32)
        etype = np.ascontiguousarray(etype, dtype=np.uint8)
        dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
        d = _abi.MapDesc(len(sx), dp(sx), dp(sy), spop.ctypes.data_as(C.POINTER(C.c_uint32)), len(ex), dp(ex), dp(ey),
                         etype.ctypes.data_as(C.POINTER(C.c_uint8)), dp(ecap), len(cx), dp(cx), dp(cy), int(grid_n),
                         float(grid_step))
        check(self.L.eg_map_set(self.h, C.byref(d)))

    def map_info(self):
        out = (C.c_uint32 * 4)()
        check(self.L.eg_map_info(self.h, out))
        return dict(n_settlements=out[0], n_existing=out[1], n_coast=out[2], grid_n=out[3])

    def site_tables(self, year_index, rclass, pclass):
        ns = self.map_info()["grid_n"] ** 2
        pref, stat, order = np.zeros(ns), np.zeros(ns), np.zeros(ns, np.uint32)
        check(self.L.eg_map_site_tables(self.h, year_index, rclass, pclass, _abi.ptr(pref), _abi.ptr(stat), _abi.ptr(order)))
        return pref, stat, order

    def site_static(self):
        ns = self.map_info()["grid_n"] ** 2
        c, o = np.zeros(ns), np.zeros(ns)
        check(self.L.eg_map_site_static(self.h, _abi.ptr(c), _abi.ptr(o)))
        return c, o

    # ---- hot path, host buffers ----
    def rollout(self, weights, n, seed=1, first_episode=0, cfg=None, want_traj=True, want_sites=False,
                want_yearly=False, out=None):
        cfg = cfg or _abi.RunCfg()
        out = out or {}
        res = out.get("results") if out.get("results") is not None else np.zeros(n, _abi.RESULT_DTYPE)
        traj = (out.get("traj") if out.get("traj") is not None else np.zeros(n, _abi.TRAJ_DTYPE)) if want_traj else None
        sites = np.zeros(n, _abi.SITES_DTYPE) if want_sites else None
        yearly = np.zeros(n, _abi.YEARLY_DTYPE) if want_yearly else None
        check(self.L.eg_rollout_batch(self.h, weights.h, C.byref(cfg), seed, first_episode, n, _abi.ptr(res),
                                      _abi.ptr(traj), _abi.ptr(sites), _abi.ptr(yearly)))
        return res, traj, sites, yearly

    def replay(self, traj_in, cfg=None, want_sites=True, want_yearly=True):
        cfg = cfg or _abi.RunCfg()
        traj_in = np.ascontiguousarray(traj_in)
        assert traj_in.dtype == _abi.TRAJ_DTYPE
        n = len(traj_in)
        res = np.zeros(n, _abi.RESULT_DTYPE)
        sites = np.zeros(n, _abi.SITES_DTYPE) if want_sites else None
        yearly = np.zeros(n, _abi.YEARLY_DTYPE) if want_yearly else None
        check(self.L.eg_replay_batch(self.h, C.byref(cfg), _abi.ptr(traj_in), n, _abi.ptr(res), _abi.ptr(sites),
                                     _abi.ptr(yearly)))
        return res, sites, yearly

    # ---- hot path, device buffers (torch uint8 tensors sized by the dtypes in _abi) ----
    def weights_upload(self, weights):
        check(self.L.eg_weights_upload(self.h, weights.h))

    def rollout_device(self, n, seed, first_episode, d_results, d_traj=None, d_sites=None, d_yearly=None, cfg=None):
        cfg = cfg or _abi.RunCfg()
        check(self.L.eg_rollout_batch_device(self.h, C.byref(cfg), seed, first_episode, n, _dev_ptr(d_results),
                                             _dev_ptr(d_traj), _dev_ptr(d_sites), _dev_ptr(d_yearly)))

    def replay_device(self, n, d_traj_in, d_results, d_sites=None, d_yearly=None, cfg=None):
        cfg = cfg or _abi.RunCfg()
        check(self.L.eg_replay_batch_device(self.h, C.byref(cfg), _dev_ptr(d_traj_in), n, _dev_ptr(d_results),
                                            _dev_ptr(d_sites), _dev_ptr(d_yearly)))

    def update_device(self, weights, n, d_results, d_traj, replay_best=False, rng_seed=0):
        """The write-lock section of multi_simulation.rs:494-508 for a batch, in episode order, on the GPU (device buffers)."""
        st = _abi.UpdateStats()
        check(self.L.eg_update_device(self.h, weights.h, _dev_ptr(d_results), _dev_ptr(d_traj), int(n), int(replay_best),
                                      int(rng_seed), C.byref(st)))
        return st

    def train_batch_inorder(self, weights, n, seed, first_episode, cfg=None, rng_seed=0):
        """Snapshot upload, rollout of n episodes from it and the in-order update, all on the GPU."""
        cfg = cfg or _abi.RunCfg()
        st = _abi.UpdateStats()
        check(self.L.eg_train_batch_inorder(self.h, weights.h, C.byref(cfg), int(seed), int(first_episode), int(n),
                                            int(rng_seed), C.byref(st)))
        return st

    def update_stats_device(self, weights, n, d_results, d_traj, d_stats, d_best_score, d_best_index):
        check(self.L.eg_update_stats_device(self.h, weights.h, _dev_ptr(d_results), _dev_ptr(d_traj), n,
                                            _dev_ptr(d_stats), _dev_ptr(d_best_score), _dev_ptr(d_best_index)))

    def update_stats_clear_device(self, d_stats):
        check(self.L.eg_update_stats_clear_device(self.h, _dev_ptr(d_stats)))

    def update_pack_best_device(self, n, d_results, d_traj, d_best_score, d_best_index, first_global_episode, d_record):
        check(self.L.eg_update_pack_best_device(self.h, _dev_ptr(d_results), _dev_ptr(d_traj), n, _dev_ptr(d_best_score),
                                                _dev_ptr(d_best_index), first_global_episode, _dev_ptr(d_record)))

    def update_pack_exchange_device(self, n, d_results, d_traj, d_stats, d_best_score, d_best_index, first_global_episode,
                                    peer_buffers, peer_flags, rank, epoch, d_error):
        """pack + all-gather over NVLink peer memory in one kernel (peer_buffers / peer_flags: lists of device addresses)"""
        world = len(peer_buffers)
        pb = (C.c_uint64 * world)(*[int(x) for x in peer_buffers])
        pf = (C.c_uint64 * world)(*[int(x) for x in peer_flags])
        check(self.L.eg_update_pack_exchange_device(self.h, _dev_ptr(d_results), _dev_ptr(d_traj), n, _dev_ptr(d_stats),
                                                    _dev_ptr(d_best_score), _dev_ptr(d_best_index), int(first_global_episode),
                                                    pb, pf, world, int(rank), int(epoch), _dev_ptr(d_error)))

    def export_best_run_csv(self, weights, output_dir, cfg=None):
        """CsvExporter::export_simulation_results for the best strategy in `weights`; returns the directory written."""
        cfg = cfg or _abi.RunCfg()
        buf = C.create_string_buffer(512)
        check(self.L.eg_export_best_run_csv(self.h, weights.h, C.byref(cfg), os.fsencode(output_dir), buf))
        return buf.value.decode()

    def location_analysis(self, use_loaded_map, half_steps=25, step=2000.0, first_point=0, n_points=None, year_index=0):
        side = 2 * half_steps + 1
        n = side * side - first_point if n_points is None else n_points
        out = np.zeros((n, _abi.N_GEN_TYPES))
        check(self.L.eg_location_analysis_year(self.h, int(use_loaded_map), int(year_index), half_steps, step, _abi.ptr(out), first_point, n))
        return out

    def location_analysis_sites(self, use_loaded_map, sites_per_axis, step, year_first=0, n_years=26, first_site=0, n_sites=None,
                                d_scores=None):
        """All candidate sites x years x 15 types in one pass (BASELINE configs[4]); returns [n_sites, n_years, 15], or
        queues the kernel into the device buffer `d_scores` and returns None."""
        n = sites_per_axis * sites_per_axis - first_site if n_sites is None else n_sites
        if d_scores is not None:
            check(self.L.eg_location_analysis_sites_device(self.h, int(use_loaded_map), sites_per_axis, float(step), year_first,
                                                           n_years, first_site, n, _dev_ptr(d_scores)))
            return None
        out = np.zeros((n, n_years, _abi.N_GEN_TYPES))
        check(self.L.eg_location_analysis_sites(self.h, int(use_loaded_map), sites_per_axis, float(step), year_first, n_years,
                                                first_site, n, _abi.ptr(out)))
        return out

    def location_analysis_write(self, use_loaded_map, min_suitability=0.3, cache_dir=None, text_path=None):
        """analyze_locations + save_cache + save_to_file (bin/analyze_locations.rs)"""
        check(self.L.eg_location_analysis_write(self.h, int(use_loaded_map), float(min_suitability),
                                                os.fsencode(cache_dir) if cache_dir else None,
                                                os.fsencode(text_path) if text_path else None))

    def train_batch_results(self, n, want_traj=True):
        """Results (and records) of the last eg_train_batch_* call, copied to the host."""
        res = np.zeros(n, _abi.RESULT_DTYPE)
        traj = np.zeros(n, _abi.TRAJ_DTYPE) if want_traj else None
        check(self.L.eg_train_batch_results(self.h, _abi.ptr(res), _abi.ptr(traj)))
        return res, traj

    def sync(self):
        check(self.L.eg_sync(self.h))

    def kernel_launches(self):
        return int(self.L.eg_kernel_launches(self.h))
