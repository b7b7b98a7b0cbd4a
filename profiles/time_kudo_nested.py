"""Time the nested Kudo assemble (srj_kudo_assemble_nested) on a seeded table of ~20 M rows:
INT64 key | LIST<INT32> | STRUCT<INT32, STRING> | map LIST<STRUCT<STRING, INT64>>, cut into 200 partitions written on
the host by the CPU restatement of the format (tests/kudo_nested_oracle.py) and uploaded.  Prints ms (CUDA events, after a warm-up),
the bytes moved (partition buffer read + every assembled buffer written), GB/s and the fraction of the 6576 GB/s copy
peak used throughout DESIGN.md, with the card name and power limit.

    python profiles/time_kudo_nested.py [rows] [partitions]
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "spark-rapids-jni_b200"), os.path.join(ROOT, "tests")]
import numpy as np
import torch

import srj_b200 as S
import kudo_nested_oracle as K
from oracle import oracle as O
from srj_b200 import _native as N

PEAK_GBS = 6576.1
n = int(sys.argv[1]) if len(sys.argv) > 1 else 20_000_000
P = int(sys.argv[2]) if len(sys.argv) > 2 else 200
rng = np.random.default_rng(20)


def mask(k, frac=0.04):
    return O.pack_mask(rng.random(k) >= frac)


def strings(k):
    lens = rng.integers(0, 13, k).astype(np.int32)
    offs = np.zeros(k + 1, np.int32)
    np.cumsum(lens, out=offs[1:])
    return O.HCol(O.STRING, rng.integers(32, 127, int(offs[-1]), dtype=np.uint8), mask(k), offs, 0, k)


def fixed(t, k):
    return O.HCol(t, rng.integers(0, 256, k * O.size_of(t), dtype=np.uint8), mask(k), None, 0, k)


def list_of(child_fn, k, max_len):
    lens = rng.integers(0, max_len + 1, k)
    offs = np.zeros(k + 1, np.int32)
    np.cumsum(lens, out=offs[1:])
    return O.HCol(O.LIST, None, mask(k), offs, 0, k, [child_fn(int(offs[-1]))])


cols = [fixed(O.INT64, n),
        list_of(lambda k: fixed(O.INT32, k), n, 4),
        O.HCol(O.STRUCT, None, mask(n), None, 0, n, [fixed(O.INT32, n), strings(n)]),
        list_of(lambda k: O.HCol(O.STRUCT, None, None, None, 0, k, [strings(k), fixed(O.INT64, k)]), n, 3)]
splits = np.linspace(0, n, P + 1).astype(np.int64).tolist()
buf_h, offs_h = K.split(cols, splits)
buf, offs = torch.from_numpy(buf_h).cuda(), torch.from_numpy(offs_h).cuda()
del buf_h

b = S.Schema.builder()
b.column(S.DType(S.DType.INT64), "key")
b.addColumn(S.DType(S.DType.LIST), "xs").column(S.DType(S.DType.INT32), "x")
b.addColumn(S.DType(S.DType.STRUCT), "s").column(S.DType(S.DType.INT32), "a").column(S.DType(S.DType.STRING), "b")
b.addColumn(S.DType(S.DType.LIST), "m").addColumn(S.DType(S.DType.STRUCT), "kv").column(S.DType(S.DType.STRING), "k").column(S.DType(S.DType.INT64), "v")
schema = b.build()

# sizes once, outputs allocated once; the timed step is srj_kudo_assemble_nested (memsets + the move kernel)
from srj_b200.kudo import KudoGpuSerializer as KS
tbl = KS.assembleFromDeviceRaw(schema, buf, offs)
lib = N.lib()
ids, nch = schema.getFlattenedTypeIds(), schema.getFlattenedNumChildren()
F = len(ids)
ws = torch.empty(lib.srj_kudo_nested_workspace_bytes(F, P), dtype=torch.uint8, device="cuda")
st = int(torch.cuda.current_stream().cuda_stream)
import ctypes as C
rows, chars = (C.c_int64 * F)(), (C.c_int64 * F)()
N.check(lib.srj_kudo_assemble_nested_sizes(buf.data_ptr(), offs.data_ptr(), P, (C.c_int32 * F)(*ids), (C.c_int32 * F)(*nch), F, rows, chars,
                                           ws.data_ptr(), st))
carr = S._carray(tbl.columns)


def step():
    N.check(lib.srj_kudo_assemble_nested(buf.data_ptr(), offs.data_ptr(), P, carr, len(tbl.columns), ws.data_ptr(), st))


def written(c):
    t = sum(x.numel() * x.element_size() for x in (c.data, c.mask, c.offsets) if x is not None)
    return t + sum(written(k) for k in ([c.child] if c.child is not None else []) + list(c.children or []))


for _ in range(3):
    step()
torch.cuda.synchronize()
k = 20
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(k):
    step()
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / k
moved = buf.numel() + sum(written(c) for c in tbl.columns)
try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30)
    card = q.stdout.strip()
except Exception:
    card = torch.cuda.get_device_name(0) + ", power limit unknown"
print(f"kudo nested assemble: rows={n} partitions={P} flattened_columns={F} buffer={buf.numel() / 1e9:.3f} GB ms={ms:.3f} "
      f"bytes_moved={moved / 1e9:.3f} GB GB/s={moved / ms / 1e6:.0f} frac_of_{PEAK_GBS:.0f}={moved / ms / 1e6 / PEAK_GBS:.3f} card=[{card}]")
