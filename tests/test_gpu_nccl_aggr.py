"""sum(rate(m[5m])) by (g) over TWO GPUs with the collective inside the library (csrc/comm.inc): one process per GPU, the NCCL
communicator is created by vmb_ctx_comm_init from a unique id passed over a pipe (no torch.distributed anywhere), the per-GPU
partial states are merged by vmb_aggr_allreduce inside vmb_eval_rollup_aggr_dist.  Both ranks must return the oracle's fold over
ALL series (aggr_incremental.go:98-168).  Needs 2 GPUs; skipped on a single-GPU machine."""
import multiprocessing as mp
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
T0 = 1_700_000_000_000
HERE = os.path.dirname(os.path.abspath(__file__))


def _make_blocks(seed, S):
    sys.path.insert(0, HERE)
    import blockgen
    rng = np.random.default_rng(seed)
    blocks = []
    for i in range(S):
        kind = ["counter", "counter_resets", "gauge"][i % 3]
        tk = "jitter" if i % 7 == 3 else "regular"  # some series take the un-fused pipeline
        blocks.append(blockgen.OBlock(blockgen.gen_timestamps(rng, tk, 2048, T0), blockgen.gen_values(rng, kind, 2048), -2, 64, i))
    return blocks


def _worker(rank, world, conn, seed, S, G, aggrs, q):
    try:
        sys.path.insert(0, HERE)
        sys.path.insert(0, os.path.dirname(HERE))
        import torch
        torch.cuda.set_device(rank)
        import blockgen
        import victoriametrics_b200 as vm
        ctx = vm.Context(rank)
        if rank == 0:
            uid = vm.Context.comm_unique_id()
            conn.send(uid)
        else:
            uid = conn.recv()
        ctx.comm_init(uid, world, rank)
        assert ctx.comm_size == world
        blocks = _make_blocks(seed, S)
        mine = [b for b in blocks if b.series_idx % world == rank]   # shard by series id (MetricID mod ngpu, SURVEY 8e)
        for k, b in enumerate(mine):
            b.series_idx = k
        groups_all = (np.arange(S) * 3 % G).astype(np.uint32)
        groups = groups_all[rank::world].copy()
        descs, payload = blockgen.to_blockset(mine)
        B = vm.storage.Blocks(descs, payload, ctx)
        start, end, step, window = T0 + 300000, T0 + 15000 * 2040, 15000, 300000
        out = {}
        for aggr in aggrs:
            func = "rate" if aggr not in ("min", "max") else "avg_over_time"
            res, _ = vm.promql.eval_rollup_aggr_dist(aggr, func, B, groups, G, start, end, step, window)
            out[aggr] = res
        ctx.comm_destroy()
        q.put((rank, out))
    except Exception as e:  # surface the failure in the parent
        import traceback
        q.put((rank, "ERROR: %r\n%s" % (e, traceback.format_exc())))


def test_two_gpu_aggregate_through_library_nccl(oracle):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import victoriametrics_b200 as vm
    from rollup_names import AGGR
    from test_baseline_configs import _oracle_rollup_matrix
    seed, S, G, world = 4711, 90, 5, 2
    aggrs = ["sum", "avg", "count", "min", "max", "sum2"]
    mpc = mp.get_context("spawn")
    a, b = mpc.Pipe()
    q = mpc.Queue()
    procs = [mpc.Process(target=_worker, args=(r, world, (a if r == 0 else b), seed, S, G, aggrs, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = {}
    for _ in range(world):
        r, out = q.get(timeout=300)
        assert not isinstance(out, str), out
        results[r] = out
    for p in procs:
        p.join(timeout=60)
    blocks = _make_blocks(seed, S)
    start, end, step, window = T0 + 300000, T0 + 15000 * 2040, 15000, 300000
    groups_all = (np.arange(S) * 3 % G).astype(np.uint32)
    for aggr in aggrs:
        func = "rate" if aggr not in ("min", "max") else "avg_over_time"
        rc = vm.promql.get_rollup_configs(func, start, end, step, window)
        rolled = _oracle_rollup_matrix(oracle, blocks, func, start, end, step, window)
        e_v, e_c = np.zeros((G, rc.points)), np.zeros((G, rc.points))
        for s in range(S):
            row = np.ascontiguousarray(rolled[s])
            g = int(groups_all[s])
            oracle.lib().vmo_aggr_update(AGGR[aggr], e_v[g].ctypes.data_as(oracle.f64p), e_c[g].ctypes.data_as(oracle.f64p),
                                         row.ctypes.data_as(oracle.f64p), rc.points)
        for g in range(G):
            oracle.lib().vmo_aggr_finalize(AGGR[aggr], e_v[g].ctypes.data_as(oracle.f64p), e_c[g].ctypes.data_as(oracle.f64p), rc.points)
        for r in range(world):
            got = results[r][aggr]
            assert np.array_equal(np.isnan(got), np.isnan(e_v)), (aggr, r)
            assert np.allclose(got, e_v, rtol=1e-12, atol=0, equal_nan=True), (aggr, r)
        assert np.array_equal(results[0][aggr].view(np.uint64), results[1][aggr].view(np.uint64)), aggr  # every rank holds the same result
