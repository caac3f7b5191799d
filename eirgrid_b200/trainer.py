"""Batch training loop: the B200 replacement of the reference's rayon loop (core/multi_simulation.rs:425-611).

One process per GPU. Each step every rank
  1. uploads the shared weights snapshot        (== local_weights = shared.read().clone(), :457-460)
  2. rolls out `episodes_per_gpu` episodes       (== run_iteration for its shard of iteration ids, :472)
  3. accumulates the update statistics on the GPU (== the write-lock section :494-508, batch-synchronous form)
  4. exchanges them: ONE NCCL all-gather of [statistics table | this rank's best episode record] (42 KB per rank);
     every rank adds the tables up in rank order (integers: the same sum everywhere) and picks the batch winner
  5. applies the identical update on every rank  (eg_update_combine_apply)

PyTorch is used for device buffers, streams and torch.distributed only.
"""
import ctypes as C
import os

import numpy as np

from . import _abi, _lib


def _torch():
    import torch
    return torch


REC_BYTES = 16 + _abi.RESULT_DTYPE.itemsize + _abi.TRAJ_DTYPE.itemsize  # [score f64 | global id i64 | eg_result | eg_traj]
assert REC_BYTES % 8 == 0


def pack_record(score, global_index, result, traj):
    """Per-rank candidate for the batch winner as a flat uint8 array."""
    rec = np.zeros(REC_BYTES, np.uint8)
    rec[0:8] = np.frombuffer(np.float64(score).tobytes(), np.uint8)
    rec[8:16] = np.frombuffer(np.int64(global_index).tobytes(), np.uint8)
    rb = _abi.RESULT_DTYPE.itemsize
    rec[16:16 + rb] = np.frombuffer(np.ascontiguousarray(result).tobytes(), np.uint8)
    rec[16 + rb:] = np.frombuffer(np.ascontiguousarray(traj).tobytes(), np.uint8)
    return rec


def combine_and_apply(weights, stats_sum, all_records, n_total, first_episode):
    """Host side of the exchange step, identical on every rank (eg_update_combine_apply): pick the batch winner among
    the per-rank candidates (highest score, lowest episode id) and apply the summed statistics to the weights.
    stats_sum: int64[STATS_WORDS] already summed over ranks; all_records: uint8[world, REC_BYTES]."""
    rec = np.ascontiguousarray(all_records, dtype=np.uint8).reshape(-1, REC_BYTES)
    stats = np.ascontiguousarray(stats_sum, dtype=np.int64)
    st = _abi.UpdateStats()
    _lib.check(_lib.lib().eg_update_combine_apply(weights.h, _abi.ptr(stats), _abi.ptr(rec), rec.shape[0], int(n_total),
                                                  int(first_episode), C.byref(st)))
    return st


PACK_WORDS = _abi.STATS_WORDS + REC_BYTES // 8  # int64 words a rank contributes to the exchange step


def shard_of(total, rank, world):
    """(first episode inside the batch, episode count) of `rank` when a batch of `total` episodes is split over `world`
    ranks: total // world each, the first total % world ranks one more (a ragged last batch never runs past the
    requested iteration count)."""
    base, rem = divmod(int(total), int(world))
    return rank * base + min(rank, rem), base + (1 if rank < rem else 0)


def pack_buffer(stats, record):
    """[statistics int64[STATS_WORDS] | candidate record] as one int64 array: what a rank sends in the exchange step."""
    out = np.zeros(PACK_WORDS, np.int64)
    out[:_abi.STATS_WORDS] = stats
    out[_abi.STATS_WORDS:] = np.ascontiguousarray(record, dtype=np.uint8).view(np.int64)
    return out


def sum_and_apply(weights, all_packs, n_total, first_episode):
    """Host side of the exchange step after the all-gather, identical on every rank: add the ranks' statistics tables up
    in rank order (integers: the same sum everywhere), pick the winner among their candidate records and apply."""
    packs = np.ascontiguousarray(all_packs, dtype=np.int64).reshape(-1, PACK_WORDS)
    stats_sum = packs[:, :_abi.STATS_WORDS].sum(axis=0, dtype=np.int64)
    records = np.ascontiguousarray(packs[:, _abi.STATS_WORDS:]).view(np.uint8)
    return combine_and_apply(weights, stats_sum, records, n_total, first_episode)


class BatchTrainer:
    def __init__(self, episodes_per_gpu, seed=1, device=None, cfg=None, weights=None, asset_dir=None, map_arrays=None,
                 distributed=None, want_sites=False):
        torch = _torch()
        if not torch.cuda.is_available():
            raise _lib.EirgridError(-4, "no CUDA device; eirgrid_b200 has no CPU fallback")
        import torch.distributed as dist
        self.dist = dist if (distributed if distributed is not None else dist.is_initialized()) else None
        self.rank = self.dist.get_rank() if self.dist else 0
        self.world = self.dist.get_world_size() if self.dist else 1
        self.device_index = int(os.environ.get("LOCAL_RANK", 0)) if device is None else int(device)
        torch.cuda.set_device(self.device_index)
        self.device = torch.device("cuda", self.device_index)
        # a dedicated (non-default) stream shared by the library's kernels, the torch copies and the collectives
        self.stream = torch.cuda.Stream(self.device)
        self.ctx = _lib.Context(self.device_index, self.stream.cuda_stream)
        assert self.stream.cuda_stream != 0
        if map_arrays is not None:
            self.ctx.map_set(*map_arrays)
        else:
            self.ctx.map_load_dir(asset_dir)
        self.n = int(episodes_per_gpu)
        self.seed = int(seed)
        self.cfg = cfg or _abi.RunCfg()
        self.weights = weights or _lib.Weights()
        self.next_episode = 0  # global id of the first episode of the next batch
        self.offset = self.rank * self.n  # this rank's first episode inside the batch
        self.n_total = self.n * self.world
        u8 = torch.uint8
        self.d_results = torch.empty(self.n * _abi.RESULT_DTYPE.itemsize, dtype=u8, device=self.device)
        self.d_traj = torch.empty(self.n * _abi.TRAJ_DTYPE.itemsize, dtype=u8, device=self.device)
        self.d_sites = torch.empty(self.n * _abi.SITES_DTYPE.itemsize, dtype=u8, device=self.device) if want_sites else None
        # what a rank contributes to the exchange step, one flat buffer: [statistics table int64[STATS_WORDS] | candidate
        # record: score f64, global index i64, eg_result, eg_traj]
        self.rec_bytes = REC_BYTES
        self.pack_words = PACK_WORDS
        self.d_pack = torch.zeros(self.pack_words, dtype=torch.int64, device=self.device)
        self.d_stats = self.d_pack[:_abi.STATS_WORDS]
        self.d_rec = self.d_pack[_abi.STATS_WORDS:].view(u8)
        self.d_best_score = torch.zeros(1, dtype=torch.float64, device=self.device)
        self.d_best_index = torch.zeros(1, dtype=torch.int64, device=self.device)
        self.d_all_pack = torch.zeros(self.world * self.pack_words, dtype=torch.int64, device=self.device)
        self.h_all_pack = torch.zeros(self.world * self.pack_words, dtype=torch.int64).pin_memory()
        self.h2d_bytes_per_step = 0
        self.d2h_bytes_per_step = self.h_all_pack.numel() * 8
        self.exchange_kind = "none" if self.world == 1 else "nccl all-gather"
        self.last_stats = None
        torch.cuda.synchronize(self.device)  # allocations above ran on the default stream

    def set_batch(self, total):
        """Split a batch of `total` episodes over the ranks: rank r takes total // world episodes, the first total % world
        ranks one more (a ragged last batch never runs past the requested iteration count). At most episodes_per_gpu each."""
        self.offset, self.n = shard_of(total, self.rank, self.world)
        assert self.n <= self.d_results.numel() // _abi.RESULT_DTYPE.itemsize, "batch larger than the buffers"
        self.n_total = int(total)

    # -- pieces (also used by bench.py to time the device-resident part alone) --
    def upload_weights(self):
        self.ctx.weights_upload(self.weights)

    def launch_rollout(self, first_episode=None):
        first = self.next_episode + self.offset if first_episode is None else first_episode
        self.ctx.rollout_device(self.n, self.seed, first, self.d_results, self.d_traj, self.d_sites, None, self.cfg)

    def launch_stats(self):
        self.ctx.update_stats_clear_device(self.d_stats)
        self.ctx.update_stats_device(self.weights, self.n, self.d_results, self.d_traj, self.d_stats, self.d_best_score,
                                     self.d_best_index)

    def _pack_best(self):
        self.ctx.update_pack_best_device(self.n, self.d_results, self.d_traj, self.d_best_score, self.d_best_index,
                                         self.next_episode + self.offset, self.d_rec)

    def exchange(self):
        """The path's only exchange step: one all-gather of every rank's [statistics | best-episode record] buffer,
        queued on the trainer's stream (a device copy when there is one rank)."""
        self._pack_best()
        with _torch().cuda.stream(self.stream):
            if self.dist and self.world > 1:
                self.dist.all_gather_into_tensor(self.d_all_pack, self.d_pack)
            else:
                self.d_all_pack.copy_(self.d_pack)

    def reduce_stats(self):
        """Exchange step of the device-resident pipeline (bench.py's `value`): winner record packed, buffers gathered."""
        self.exchange()

    def check_exchange(self):
        """No-op: NCCL reports a failed all-gather itself. Kept for callers that check after every exchange step."""

    def warm_exchange(self):
        """Run the gather / copy part of step() once without applying anything (warm-up)."""
        self.exchange()
        with _torch().cuda.stream(self.stream):
            self.h_all_pack.copy_(self.d_all_pack, non_blocking=True)
        self.stream.synchronize()

    def step(self):
        """One training batch through the public path: weights in from the host, update statistics back."""
        torch = _torch()
        self.upload_weights()
        self.launch_rollout()
        self.launch_stats()
        self.exchange()
        with torch.cuda.stream(self.stream):
            self.h_all_pack.copy_(self.d_all_pack, non_blocking=True)
        self.stream.synchronize()
        n_total = self.n_total
        st = sum_and_apply(self.weights, self.h_all_pack.numpy(), n_total, self.next_episode)
        self.next_episode += n_total
        self.last_stats = st
        return st

    def step_inorder(self, n=None, rng_seed=0):
        """One batch under the reference's own rule: `n` episodes (default episodes_per_gpu) sampled from one snapshot, then
        the per-episode update in episode order on the GPU (eg_train_batch_inorder; learning.rs:131-373 applied by
        csrc/update.cu). The rule is sequential in the episodes, so under several ranks every rank runs the SAME episodes
        and ends with the same table without an exchange (replicas)."""
        n = self.n if n is None else int(n)
        st = self.ctx.train_batch_inorder(self.weights, n, self.seed, self.next_episode, self.cfg, rng_seed)
        self.next_episode += n
        self.last_stats = st
        return st

    def step_inorder_sharded(self, total=None, rng_seed=0):
        """The reference's rule on several GPUs: the batch's episodes are rolled out in shards (rank r takes its slice of the
        ids, like step()), every rank's results and action records are all-gathered over NVLink (1,152 B per episode), and
        every rank then applies the per-episode update to the whole batch in episode order on its own GPU
        (eg_update_device) — the rule is sequential in the episodes, so the update itself is replicated, identical inputs
        giving identical tables without a further exchange. With one rank this is step_inorder()."""
        torch = _torch()
        total = self.n_total if total is None else int(total)
        if not (self.dist and self.world > 1):
            return self.step_inorder(total, rng_seed=rng_seed)
        self.set_batch(total)
        slot = shard_of(total, 0, self.world)[1]  # the largest shard: the gather moves equal slots
        rb, tb = _abi.RESULT_DTYPE.itemsize, _abi.TRAJ_DTYPE.itemsize
        if getattr(self, "_gather_slot", 0) < slot:
            self.d_all_results = torch.empty(self.world * slot * rb, dtype=torch.uint8, device=self.device)
            self.d_all_traj = torch.empty(self.world * slot * tb, dtype=torch.uint8, device=self.device)
            self._gather_slot = slot
        self.upload_weights()
        self.launch_rollout()
        with torch.cuda.stream(self.stream):
            self.dist.all_gather_into_tensor(self.d_all_results[:self.world * slot * rb], self.d_results[:slot * rb])
            self.dist.all_gather_into_tensor(self.d_all_traj[:self.world * slot * tb], self.d_traj[:slot * tb])
            if total % self.world:  # ragged: the shorter shards leave a hole at the end of their slot; close the gaps
                res = torch.cat([self.d_all_results[r * slot * rb:(r * slot + shard_of(total, r, self.world)[1]) * rb] for r in range(self.world)])
                traj = torch.cat([self.d_all_traj[r * slot * tb:(r * slot + shard_of(total, r, self.world)[1]) * tb] for r in range(self.world)])
            else:
                res, traj = self.d_all_results, self.d_all_traj
        st = self.ctx.update_device(self.weights, total, res, traj, replay_best=bool(self.cfg.replay_best), rng_seed=rng_seed)
        self.next_episode += total
        self.last_stats = st
        return st

    def fetch_results(self):
        """Copy this rank's last batch to the host as structured arrays (results, trajectories)."""
        self.stream.synchronize()
        with _torch().cuda.stream(self.stream):
            res = self.d_results[:self.n * _abi.RESULT_DTYPE.itemsize].cpu().numpy().view(_abi.RESULT_DTYPE)
            traj = self.d_traj[:self.n * _abi.TRAJ_DTYPE.itemsize].cpu().numpy().view(_abi.TRAJ_DTYPE)
        return res, traj

    def close(self):
        self.ctx.close()
