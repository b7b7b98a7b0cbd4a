"""GPU tests of the nested Kudo assemble (csrc/kudo.cu over srj_kudo_assemble_nested_sizes / srj_kudo_assemble_nested,
KudoGpuSerializer.assembleFromDeviceRaw with a Schema): partitions written by the CPU restatement of the nested format
(tests/kudo_nested_oracle.py) assembled on the device equal the input table and, bit for bit, the oracle's assembly --
for the tables of the reference's tests under every slicing, the two merge known answers, seeded random trees, and
malformed input."""
import ctypes as C
import struct

import numpy as np
import pytest
import torch

import kudo_nested_oracle as K
from golden import kudo_nested_golden as G
from oracle import oracle as O
from util import cols_equal, random_table

pytestmark = pytest.mark.gpu


def _gpu():
    import gpu_util
    gpu_util.require_cuda()
    return gpu_util


# ---- helpers: device trees to host, equality, schema ----------------------------------------------------------------
def to_host(c) -> O.HCol:
    """A device column tree (LIST `child`, STRUCT `children`) as an oracle HCol tree."""
    import srj_b200 as S
    t = c.dtype.type_id
    mask = c.mask.cpu().numpy().view(np.uint32) if c.mask is not None else None
    if t == S.DType.LIST:
        return O.HCol(t, None, mask, c.offsets.cpu().numpy(), 0, c.size, [to_host(c.child)])
    if t == S.DType.STRUCT:
        return O.HCol(t, None, mask, None, 0, c.size, [to_host(k) for k in (c.children or [])])
    d, m, o = c.to_numpy()
    if d is None:
        d = np.zeros(0, np.uint8)
    return O.HCol(t, d, m, o, c.dtype.scale, c.size)


def tree_equal(a: O.HCol, b: O.HCol) -> bool:
    """Same type, rows and validity; LIST / STRING offsets identical; children equal; leaf values equal where valid."""
    if a.type_id != b.type_id or a.size != b.size or not np.array_equal(a.valid(), b.valid()):
        return False
    if a.type_id == O.LIST:
        return np.array_equal(a.offsets, b.offsets) and tree_equal(a.children[0], b.children[0])
    if a.type_id == O.STRUCT:
        return len(a.children or []) == len(b.children or []) and all(tree_equal(x, y) for x, y in zip(a.children or [], b.children or []))
    if a.type_id == O.STRING and not np.array_equal(a.offsets, b.offsets):
        return False
    return cols_equal(a, b)


def tree_bits_equal(a: O.HCol, b: O.HCol) -> bool:
    """Bit-exact: valid bits, offsets and every data byte (null payloads included)."""
    if a.type_id != b.type_id or a.size != b.size or not np.array_equal(a.valid(), b.valid()):
        return False
    if a.offsets is not None or b.offsets is not None:
        if not np.array_equal(np.asarray(a.offsets)[:a.size + 1], np.asarray(b.offsets)[:b.size + 1]):
            return False
    if a.type_id in (O.LIST, O.STRUCT):
        return len(a.children or []) == len(b.children or []) and all(tree_bits_equal(x, y) for x, y in zip(a.children or [], b.children or []))
    n = int(a.offsets[a.size]) if a.type_id == O.STRING else a.size * O.size_of(a.type_id)
    return np.array_equal(np.ascontiguousarray(a.data).view(np.uint8)[:n], np.ascontiguousarray(b.data).view(np.uint8)[:n])


def schema_of(cols):
    import srj_b200 as S
    b = S.Schema.builder()

    def add(builder, c, name):
        if c.type_id in (O.LIST, O.STRUCT):
            child = builder.addColumn(S.DType(c.type_id), name)
            for i, k in enumerate(c.children or []):
                add(child, k, f"{name}.{i}")
        else:
            builder.column(S.DType(c.type_id, c.scale), name)
    for i, c in enumerate(cols):
        add(b, c, f"c{i}")
    return b.build()


def _dev(buf, offs):
    return torch.from_numpy(np.ascontiguousarray(buf)).cuda(), torch.from_numpy(np.ascontiguousarray(offs)).cuda()


def assemble_and_check(cols, buf, offs, want=None):
    """Assemble on the device; the result equals `want` (default: the oracle's assembly) and is bit-exact against the
    oracle's assembly."""
    _gpu()
    from srj_b200.kudo import KudoGpuSerializer as KS
    ids, nch, scales = K.flatten(cols)
    ref = K.assemble_nested(buf, offs, ids, nch, scales)
    tbl = KS.assembleFromDeviceRaw(schema_of(cols), *_dev(buf, offs))
    got = [to_host(c) for c in tbl.columns]
    assert len(got) == len(ref)
    for i, (g, r) in enumerate(zip(got, ref)):
        assert tree_bits_equal(g, r), f"column {i} vs the oracle"
        if want is not None:
            assert tree_equal(g, want[i]), f"column {i} vs the expected table"
    return got


def _concat(pieces):
    buf = np.concatenate(pieces) if pieces else np.zeros(0, np.uint8)
    offs = np.zeros(len(pieces) + 1, np.int64)
    np.cumsum([len(p) for p in pieces], out=offs[1:])
    return buf, offs


# ---- random trees ---------------------------------------------------------------------------------------------------
MAP = ("LIST", ("STRUCT", [O.STRING, O.INT64]))
SPECS = [
    O.INT32, O.DECIMAL128, O.STRING,
    MAP,
    ("LIST", ("LIST", O.INT8)),
    ("STRUCT", [("LIST", O.INT16), O.DECIMAL128]),
    ("STRUCT", []),
    ("STRUCT", [O.BOOL8, ("STRUCT", [O.STRING, ("LIST", O.DECIMAL128)])]),
    ("LIST", ("STRUCT", [])),
    ("LIST", O.STRING),
]


def rand_col(spec, n, rng) -> O.HCol:
    seed = int(rng.integers(1 << 30))
    nullable = rng.random() < 0.7
    valid = (rng.random(n) >= 0.25) if nullable else np.ones(n, bool)
    mask = O.pack_mask(valid) if nullable else None
    if isinstance(spec, tuple) and spec[0] == "LIST":
        lens = rng.integers(0, 5, n)                                  # empty lists included
        lens[~valid & (rng.random(n) < 0.5)] = 0                      # null lists with and without elements
        offs = np.zeros(n + 1, np.int32)
        np.cumsum(lens, out=offs[1:])
        return O.HCol(O.LIST, None, mask, offs, 0, n, [rand_col(spec[1], int(offs[-1]), rng)])
    if isinstance(spec, tuple):
        return O.HCol(O.STRUCT, None, mask, None, 0, n, [rand_col(f, n, rng) for f in spec[1]])
    return random_table([spec], n, seed=seed, null_frac=0.2 if nullable else 0.0)[0]


def rand_table(n, seed, specs=SPECS):
    rng = np.random.default_rng(seed)
    return [rand_col(s, n, rng) for s in specs]


def rand_splits(n, P, rng):
    cuts = sorted(rng.integers(0, n + 1, P - 1).tolist())             # repeats = empty partitions, unaligned starts
    return [0] + cuts + [n]


# ---- tests ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(G.GOLDEN_TABLES))
def test_golden_tables_every_slicing(name):
    build, slicings = G.GOLDEN_TABLES[name]
    t = build()
    for splits in slicings(t[0].size):
        assemble_and_check(t, *K.split(t, splits), want=t)


@pytest.mark.parametrize("case", [G.merge_list_case, G.merge_complex_struct_list_case])
def test_merge_known_answers(case):
    pieces, want = case()
    buf, offs = _concat([np.frombuffer(K.write_partition(t, off, n), np.uint8) for t, off, n in pieces])
    assemble_and_check(want, buf, offs, want=want)


@pytest.mark.parametrize("seed", range(6))
def test_random_trees(seed):
    rng = np.random.default_rng(100 + seed)
    n = int(rng.integers(1, 3000))
    t = rand_table(n, seed)
    assemble_and_check(t, *K.split(t, rand_splits(n, int(rng.integers(1, 40)), rng)), want=t)
    assemble_and_check(t, *K.split(t, [0, n]), want=t)


def test_partitions_of_two_tables():
    a, b = rand_table(1500, 1), rand_table(900, 2)
    ba, oa = K.split(a, [0, 333, 1500])
    bb, ob = K.split(b, [0, 5, 5, 900])
    buf, offs = _concat([ba[oa[1]:oa[2]], bb[ob[2]:ob[3]], bb[ob[1]:ob[2]], ba[oa[0]:oa[1]]])
    got = assemble_and_check(a, buf, offs)
    assert got[0].size == (1500 - 333) + (900 - 5) + 333


def test_two_million_rows_in_200_partitions():
    n = 2_000_000
    t = rand_table(n, 7, specs=[O.INT64, ("LIST", O.INT32), ("STRUCT", [O.INT32, O.STRING]), MAP])
    splits = np.linspace(0, n, 201).astype(np.int64).tolist()
    assemble_and_check(t, *K.split(t, splits), want=t)


def test_flat_schema_through_the_nested_entry_points():
    """A flat schema assembled by the nested entry points gives the bytes of the flat ones."""
    G_ = _gpu()
    import srj_b200 as S
    from srj_b200.kudo import KudoGpuSerializer as KS
    types = [O.INT32, O.STRING, O.INT64, O.DECIMAL128, O.INT8, O.STRING, O.FLOAT64, O.BOOL8]
    cols = random_table(types, 5000, seed=3)
    buf, offs = _dev(*K.split(cols, [0, 0, 17, 2500, 2501, 5000]))
    flat = KS.assembleFromDeviceRaw([S.DType(t) for t in types], buf, offs)
    nested = KS.assembleFromDeviceRaw(schema_of(cols), buf, offs)
    for f, g in zip(flat.columns, nested.columns):
        hf, hg = G_.to_host(f), to_host(g)
        assert tree_bits_equal(hf, hg)
        assert np.array_equal(f.mask.cpu().numpy()[: (f.size + 31) // 32], g.mask.cpu().numpy()[: (g.size + 31) // 32])


# ---- rejections -----------------------------------------------------------------------------------------------------
def _raw_sizes(buf, offs, ids, nch):
    """srj_kudo_assemble_nested_sizes on a raw flattened schema -> status."""
    from srj_b200 import _native as N
    lib = N.lib()
    F = len(ids)
    d_buf, d_offs = _dev(buf, offs)
    ws = torch.empty(lib.srj_kudo_nested_workspace_bytes(F, len(offs) - 1), dtype=torch.uint8, device="cuda")
    rows, chars = (C.c_int64 * max(F, 1))(), (C.c_int64 * max(F, 1))()
    rc = lib.srj_kudo_assemble_nested_sizes(d_buf.data_ptr(), d_offs.data_ptr(), len(offs) - 1, (C.c_int32 * max(F, 1))(*ids),
                                            (C.c_int32 * max(F, 1))(*nch), F, rows, chars, ws.data_ptr(), int(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return rc, list(rows)[:F]


def test_rejections():
    _gpu()
    import srj_b200 as S
    from srj_b200 import _native as N
    from srj_b200.kudo import KudoGpuSerializer as KS
    t = G.build_simple_table()
    ids, nch, _ = K.flatten(t)
    buf, offs = K.split(t, [0, 2, 4])
    assert _raw_sizes(buf, offs, ids, nch) == (N.SRJ_OK, [4, 4, 4, 9, 4, 4, 4])
    # column-count mismatch: the schema without the STRUCT's last field
    with pytest.raises(S.CudfException):
        KS.assembleFromDeviceRaw(schema_of(t[:3] + [O.HCol(O.STRUCT, None, None, None, 0, 4, t[3].children[:1])]), *_dev(buf, offs))
    # a partition cut 4 bytes short through its offsets table (the allocation itself is intact)
    whole = np.frombuffer(K.write_partition(t, 0, 4), np.uint8).copy()
    _, _, _, vlen, olen, _, _ = struct.unpack(">7i", whole[:28].tobytes())
    short = np.array([0, K.header_size(len(ids)) + vlen + olen - 4], np.int64)
    assert _raw_sizes(whole, np.array([0, len(whole)], np.int64), ids, nch)[0] == N.SRJ_OK
    assert _raw_sizes(whole, short, ids, nch)[0] == N.SRJ_EINVAL
    with pytest.raises(S.CudfException):
        KS.assembleFromDeviceRaw(schema_of(t), *_dev(whole, short))
    # decreasing list offsets: the list's off[n] below off[0]
    one = np.frombuffer(K.write_partition([t[2]], 0, 4), np.uint8).copy()
    hs = K.header_size(2)
    vlen = int.from_bytes(one[12:16].tobytes(), "big")
    o_at = hs + vlen
    one[o_at + 16:o_at + 20] = np.frombuffer(np.int32(-1).tobytes(), np.uint8)     # off[4] = -1 < off[0] = 0
    assert _raw_sizes(one, np.array([0, len(one)], np.int64), [O.LIST, O.INT32], [1, 0])[0] == N.SRJ_EINVAL
    # more than 256 flattened columns
    assert _raw_sizes(buf, offs, [O.INT8] * 257, [0] * 257)[0] == N.SRJ_EUNSUPPORTED
    # a LIST without exactly one child
    assert _raw_sizes(buf, offs, [O.LIST, O.INT32, O.INT32], [2, 0, 0])[0] == N.SRJ_EINVAL
    assert _raw_sizes(buf, offs, [O.LIST], [0])[0] == N.SRJ_EINVAL


def test_list_elements_beyond_int32_overflow():
    """Two partitions of one LIST<INT8> row each, 1.1 G elements apiece (real bytes, so no read leaves the buffer):
    the assembled child would exceed INT32_MAX rows."""
    _gpu()
    import srj_b200 as S
    from srj_b200.kudo import KudoGpuSerializer as KS
    m = 1_100_000_000
    hs = K.header_size(2)
    vlen = K._pad4(hs) - hs                                            # no validity, padding only
    olen, dlen = 8, K._pad4(m)
    head = np.frombuffer(np.array([K.MAGIC, 0, 1, vlen, olen, vlen + olen + dlen, 2], ">i4").tobytes() + bytes(1 + vlen), np.uint8)
    body = np.frombuffer(np.array([0, m], "<i4").tobytes(), np.uint8)
    part = hs + vlen + olen + dlen
    buf = torch.zeros(2 * part, dtype=torch.uint8, device="cuda")
    for p in range(2):
        buf[p * part:p * part + hs + vlen] = torch.from_numpy(head.copy()).cuda()
        buf[p * part + hs + vlen:p * part + hs + vlen + 8] = torch.from_numpy(body.copy()).cuda()
    offs = torch.tensor([0, part, 2 * part], dtype=torch.int64, device="cuda")
    b = S.Schema.builder()
    b.addColumn(S.DType(S.DType.LIST), "xs").column(S.DType(S.DType.INT8), "x")
    with pytest.raises(S.CudfColumnSizeOverflowException):
        KS.assembleFromDeviceRaw(b.build(), buf, offs)
    del buf
    torch.cuda.empty_cache()
