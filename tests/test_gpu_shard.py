"""Multi-GPU configuration on real GPUs (needs >= 2; skipped on a 1-GPU box): every rank converts its contiguous row
range with the CUDA path straight into its packed slab, ONE NCCL all-gather, srj_shard_rebase_offsets -- and the
gathered chunks must equal the oracle's conversion of the whole table."""
import os
import socket
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, nrows, q):
    for p in (ROOT, os.path.join(ROOT, "spark-rapids-jni_b200"), os.path.join(ROOT, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import srj_b200 as S
        from oracle import oracle as O
        from srj_b200 import sharding
        from util import random_table
        import gpu_util as G
        types = [O.INT32, O.INT64, O.DECIMAL128, O.STRING] * 16 + [O.BOOL8, O.STRING]     # wide path (17 STRING columns)
        cols = random_table(types, nrows, seed=31)
        (offs, data), = O.convert_to_rows(cols)
        want, _ = O.convert_from_rows(data, offs, nrows, types)
        per = nrows // world
        r0, r1 = rank * per, (rank + 1) * per
        b0, b1 = sharding.rows_byte_range(offs, r0, r1)
        vec = G.rows_to_device((offs[r0:r1 + 1] - offs[r0]).astype(np.int32), data[b0:b1])
        cap = sum((len(c.data) + 15) & ~15 for c in want if c.type_id == O.STRING)
        dts = [S.DType(t) for t in types]
        lay = sharding.SlabLayout([d.size_in_bytes() for d in dts], per, cap)
        slab = torch.zeros(lay.nbytes, dtype=torch.uint8, device="cuda")
        sharding.convert_from_rows_into_slab(vec, dts, lay, slab)
        gathered, _ = sharding.gather_slab(dist, slab, world)
        tot = sharding.rebase_gathered_offsets(gathered, lay, world).cpu().numpy()
        g2 = gathered.cpu().numpy().reshape(world, lay.nbytes)
        ok = True
        for i, c in enumerate(want):
            m = np.concatenate([g2[r, lay.at_mask[i]: lay.at_mask[i] + lay.words * 4].view(np.uint32) for r in range(world)])
            ok &= np.array_equal(m, c.mask)
            if c.type_id == O.STRING:
                o = [g2[r, lay.at_data[i]: lay.at_data[i] + (per + 1) * 4].view(np.int32) for r in range(world)]
                ok &= np.array_equal(np.concatenate([o[0]] + [x[1:] for x in o[1:]]), c.offsets)
                chars = []
                for r in range(world):
                    a = lay.chars_offsets([int(tot[r, j]) for j in lay.string_cols])[lay.string_cols.index(i)]
                    chars.append(g2[r, a: a + int(tot[r, i])])
                ok &= np.array_equal(np.concatenate(chars), c.data)
            else:
                w = O.size_of(c.type_id)
                d = np.concatenate([g2[r, lay.at_data[i]: lay.at_data[i] + per * w] for r in range(world)])
                ok &= np.array_equal(d, np.ascontiguousarray(c.data).view(np.uint8))
        q.put((rank, bool(ok)))
    finally:
        dist.destroy_process_group()


def test_two_gpu_shards_allgather_equals_oracle():
    assert torch.cuda.is_available(), "CUDA device required for -m gpu tests"
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    world, nrows = 2, 4096
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, nrows, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=300) for _ in range(world)]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert all(ok for _, ok in res)


def test_slab_conversion_single_gpu():
    """The shard conversion into a packed slab + the rebase kernel on one GPU (world 1 = identity; world 2 emulated by
    converting both halves on the same device and concatenating the slabs)."""
    assert torch.cuda.is_available(), "CUDA device required for -m gpu tests"
    for p in (ROOT, os.path.join(ROOT, "spark-rapids-jni_b200"), os.path.join(ROOT, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import srj_b200 as S
    from oracle import oracle as O
    from srj_b200 import sharding
    from util import random_table
    import gpu_util as G
    types = [O.INT32, O.STRING, O.INT64, O.DECIMAL128, O.STRING, O.BOOL8] * 3
    nrows, world = 2048, 2
    cols = random_table(types, nrows, seed=32)
    (offs, data), = O.convert_to_rows(cols)
    want, _ = O.convert_from_rows(data, offs, nrows, types)
    per = nrows // world
    dts = [S.DType(t) for t in types]
    cap = sum((len(c.data) + 15) & ~15 for c in want if c.type_id == O.STRING)
    lay = sharding.SlabLayout([d.size_in_bytes() for d in dts], per, cap)
    gathered = torch.zeros(world * lay.nbytes, dtype=torch.uint8, device="cuda")
    for r in range(world):
        r0, r1 = r * per, (r + 1) * per
        b0, b1 = sharding.rows_byte_range(offs, r0, r1)
        vec = G.rows_to_device((offs[r0:r1 + 1] - offs[r0]).astype(np.int32), data[b0:b1])
        sharding.convert_from_rows_into_slab(vec, dts, lay, gathered[r * lay.nbytes:(r + 1) * lay.nbytes])
    sharding.rebase_gathered_offsets(gathered, lay, world)
    g2 = gathered.cpu().numpy().reshape(world, lay.nbytes)
    for i, c in enumerate(want):
        if c.type_id == O.STRING:
            o = [g2[r, lay.at_data[i]: lay.at_data[i] + (per + 1) * 4].view(np.int32) for r in range(world)]
            assert np.array_equal(np.concatenate([o[0]] + [x[1:] for x in o[1:]]), c.offsets), f"offsets, column {i}"
        else:
            w = O.size_of(c.type_id)
            d = np.concatenate([g2[r, lay.at_data[i]: lay.at_data[i] + per * w] for r in range(world)])
            assert np.array_equal(d, np.ascontiguousarray(c.data).view(np.uint8)), f"column {i}"
