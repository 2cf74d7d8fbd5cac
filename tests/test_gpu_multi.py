"""Multi-GPU PageRank (1-D edge-cut, one process per GPU, NCCL) against the oracle.  Needs >= 2 GPUs and
skips on a machine with one; run with `python -m pytest tests/test_gpu_multi.py -m gpu`."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, scale, exchange, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import graph_b200 as gb
        from graph_b200.multigpu import ShardedPageRank
        gb.set_device(rank)
        g = gb.DiGraph.rmat(scale, seed=42, layout=gb.Layout.Sorted)
        spr = ShardedPageRank(g, exchange=exchange)
        out = []
        for maxit, tol in ((20, 0.0), (60, 1e-5)):
            spr.run(maxit, 0.85, tol)
            out.append((spr.ran_iterations, spr.error, spr.scores_host()))
        single = g.page_rank(max_iterations=20, tolerance=0.0, mode="jacobi").scores() if rank == 0 else None
        if rank == 0:
            q.put((spr.exchange, spr.multicast, out, single))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("exchange", ["allgather", "peer"])
def test_sharded_page_rank_matches_oracle(exchange):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import oracle
    scale, world = 16, 2
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.SimpleQueue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, scale, exchange, q)) for r in range(world)]
    for p in procs:
        p.start()
    used, multicast, out, single = q.get()
    for p in procs:
        p.join(timeout=300)
        assert p.exitcode == 0
    assert used == exchange
    src, dst = oracle.rmat_edges(scale, seed=42)
    n = 1 << scale
    out_off, _ = oracle.csr_build(src, dst, n, oracle.OUTGOING, oracle.SORTED)
    in_off, in_tgt = oracle.csr_build(src, dst, n, oracle.INCOMING, oracle.SORTED)
    for (maxit, tol), (it, err, scores) in zip(((20, 0.0), (60, 1e-5)), out):
        want, wit, werr = oracle.page_rank_jacobi(in_off, in_tgt, out_off, maxit, tol, 0.85, acc64=True)
        assert it == wit
        assert np.max(np.abs(scores - want) / want) <= 1e-6
        assert abs(err - werr) <= 2e-6
    assert np.max(np.abs(out[0][2] - single) / single) <= 1e-6


def _wcc_worker(rank, world, port, scale, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import graph_b200 as gb
        from graph_b200.multigpu import ShardedWcc
        gb.set_device(rank)
        g = gb.DiGraph.rmat(scale, seed=42, layout=gb.Layout.Sorted)
        comp = ShardedWcc(g).run().cpu().numpy().view(np.uint32)
        single = g.wcc().components()
        q.put((rank, bool((comp == single).all()), int(len(np.unique(comp)))))
    finally:
        dist.destroy_process_group()


def test_sharded_wcc_bit_equal_to_single_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    scale, world = 20, 2
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.SimpleQueue()
    procs = [ctx.Process(target=_wcc_worker, args=(r, world, port, scale, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = [q.get() for _ in range(world)]
    for p in procs:
        p.join(timeout=300)
        assert p.exitcode == 0
    assert all(ok for _, ok, _ in got) and len({c for _, _, c in got}) == 1


def test_single_process_communicator_two_gpus():
    """gb_comm_* / gb_page_rank_multi: one host thread drives both devices (no torch.distributed, no
    NCCL); ranks <= 1e-6 of the oracle and of a 1-GPU run, also with early stopping."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import oracle
    import graph_b200 as gb
    scale = 16
    graphs = []
    for d in (0, 1):
        gb.set_device(d)
        graphs.append(gb.DiGraph.rmat(scale, seed=42, layout=gb.Layout.Sorted))
    gb.set_device(0)
    comm = gb.Comm([0, 1])
    src, dst = oracle.rmat_edges(scale, seed=42)
    n = 1 << scale
    out_off, _ = oracle.csr_build(src, dst, n, oracle.OUTGOING, oracle.SORTED)
    in_off, in_tgt = oracle.csr_build(src, dst, n, oracle.INCOMING, oracle.SORTED)
    for maxit, tol in ((20, 0.0), (60, 1e-5)):
        want, wit, werr = oracle.page_rank_jacobi(in_off, in_tgt, out_off, maxit, tol, 0.85, acc64=True)
        for _ in range(2):      # a second call reuses the communicator's buffers and sequence numbers
            pr = comm.page_rank(graphs, max_iterations=maxit, tolerance=tol)
            assert pr.ran_iterations == wit
            assert np.max(np.abs(pr.scores() - want) / want) <= 1e-6
            assert abs(pr.error - werr) <= 2e-6
    single = graphs[0].page_rank(max_iterations=20, tolerance=0.0, mode="jacobi").scores()
    multi = comm.page_rank(graphs, max_iterations=20, tolerance=0.0).scores()
    assert np.max(np.abs(multi - single) / single) <= 1e-6
