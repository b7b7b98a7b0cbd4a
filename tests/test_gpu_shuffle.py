"""The shuffle exchange on real GPUs over NCCL (srj_b200.shuffle.ShuffleExchange: hash partition -> Kudo split ->
all_to_all_single -> assemble).  World 1 runs on any box (the collective degenerates to a copy); world 2 needs two GPUs
and is skipped otherwise.  Expected result from the CPU oracle."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, k, q):
    for p in (ROOT, os.path.join(ROOT, "spark-rapids-jni_b200"), os.path.join(ROOT, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import gpu_util as G
        from oracle import oracle as O
        from srj_b200.shuffle import ShuffleExchange
        from util import cols_equal, random_table
        types = [O.INT32, O.STRING, O.INT64, O.DECIMAL128, O.INT8]
        P = world * k
        tables = [random_table(types, 20_000 + 1111 * r, seed=70 + r) for r in range(world)]
        out = ShuffleExchange().shuffle(G.table_to_device(tables[rank]), [0, 2], parts_per_rank=k)
        torch.cuda.synchronize()
        want = []
        for r in range(world):
            ids = O.partition_ids([tables[r][0], tables[r][2]], P)
            rc, ro, _ = O.stable_partition(tables[r], ids, P)
            want.append([O.take(c, np.arange(int(ro[rank * k]), int(ro[(rank + 1) * k]))) for c in rc])
        ok = True
        for ci, g in enumerate(out.columns):
            h = G.to_host(g)
            at = 0
            for piece in (w[ci] for w in want):
                ok &= cols_equal(O.take(h, np.arange(at, at + piece.size)), piece)
                at += piece.size
            ok &= at == h.size
        q.put((rank, bool(ok), out.getRowCount()))
    finally:
        dist.destroy_process_group()


def _run(world, k):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, k, q)) for r in range(world)]
    [p.start() for p in procs]
    res = [q.get(timeout=300) for _ in range(world)]
    [p.join(timeout=60) for p in procs]
    assert all(ok for _, ok, _ in res), res
    assert sum(n for _, _, n in res) == sum(20_000 + 1111 * r for r in range(world))


def test_shuffle_exchange_world_1():
    if not torch.cuda.is_available():
        pytest.fail("CUDA device required")
    _run(1, 5)


def test_shuffle_exchange_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _run(2, 3)
