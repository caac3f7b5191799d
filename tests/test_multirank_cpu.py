"""world_size-2 gloo test of the multi-rank exchange step on the CPU: episode-id sharding (ragged), the one all-gather of
[statistics | best-episode record], batch-winner selection and the identical host-side apply. The device-side statistics are replaced by
their numpy restatement (tests/stats_ref.py), everything after them is the product's own host code."""
import os
import socket
import sys

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _best_lists(w):
    has, b, d = w.best()
    return [x.tolist() for x in b], [x.tolist() for x in d]


def _setup_weights():
    """A snapshot with a best strategy so that the contrast statistics are non-trivial."""
    import oracle_lib as O
    from eirgrid_b200 import _lib
    world = O.World.ireland(fast=True)
    ow, gw = O.Weights(), _lib.Weights()
    res, traj, _, _ = world.rollout(ow, 24, seed=5, threads=2)
    ow.update(res, traj)
    gw.update(res, traj)
    return world, ow, gw


def _one_step(gw, ow, world, first, n_total, rank, world_size, use_dist):
    import stats_ref
    from eirgrid_b200 import trainer as T
    offset, n_per_rank = T.shard_of(n_total, rank, world_size)
    lo = first + offset
    res, traj, _, _ = world.rollout(ow, n_per_rank, seed=77, first_episode=lo, threads=2)
    t = gw.table()
    consts = stats_ref.contrast_consts(t)
    best, best_def = _best_lists(gw)
    stats, scores, _ = stats_ref.batch_stats(res, traj, consts, best, best_def)
    k = int(np.lexsort((np.arange(n_per_rank), -scores))[0])
    rec = T.pack_record(scores[k], lo + k, res[k:k + 1], traj[k:k + 1])
    pack = torch.from_numpy(T.pack_buffer(stats, rec))
    all_packs = torch.zeros(world_size * T.PACK_WORDS, dtype=torch.int64)
    if use_dist:
        dist.all_gather_into_tensor(all_packs, pack)  # the path's one exchange step
    else:
        all_packs[:] = pack
    return T.sum_and_apply(gw, all_packs.numpy(), n_total, first)


def _worker(rank, world_size, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    world, ow, gw = _setup_weights()
    first = 1000
    for step in range(2):
        st = _one_step(gw, ow, world, first, 65, rank, world_size, True)  # ragged: 33 + 32 episodes
        ow.set_table(gw.table())  # sampling weights for the next batch follow the product's update
        first += 65
    np.save(os.path.join(out_dir, "rank%d.npy" % rank), np.frombuffer(bytes(gw.table()), np.uint8))
    np.save(os.path.join(out_dir, "iwi%d.npy" % rank), np.array([st.iterations_without_improvement, st.n_improvements, st.batch_best_episode]))
    dist.destroy_process_group()


def test_two_ranks_match_one_rank(tmp_path):
    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0 = np.load(tmp_path / "rank0.npy")
    r1 = np.load(tmp_path / "rank1.npy")
    assert np.array_equal(r0, r1), "ranks diverged"
    # single process over the same 65-episode batches
    world, ow, gw = _setup_weights()
    first = 1000
    for step in range(2):
        import stats_ref
        from eirgrid_b200 import trainer as T
        res, traj, _, _ = world.rollout(ow, 65, seed=77, first_episode=first, threads=2)
        t = gw.table()
        consts = stats_ref.contrast_consts(t)
        best, best_def = _best_lists(gw)
        stats, scores, _ = stats_ref.batch_stats(res, traj, consts, best, best_def)
        k = int(np.lexsort((np.arange(65), -scores))[0])
        rec = T.pack_record(scores[k], first + k, res[k:k + 1], traj[k:k + 1])
        T.combine_and_apply(gw, stats, rec, 65, first)
        ow.set_table(gw.table())
        first += 65
    single = np.frombuffer(bytes(gw.table()), np.uint8)
    assert np.array_equal(single, r0), "2-rank result differs from the 1-rank result"


def test_shard_of_covers_the_batch_without_gaps():
    from eirgrid_b200 import trainer as T
    for total, world in ((65, 2), (100000, 8), (7, 8), (0, 4), (65536, 1)):
        shards = [T.shard_of(total, r, world) for r in range(world)]
        assert shards[0][0] == 0 and sum(n for _, n in shards) == total
        assert all(shards[r][0] + shards[r][1] == shards[r + 1][0] for r in range(world - 1))
        assert max(n for _, n in shards) - min(n for _, n in shards) <= 1
