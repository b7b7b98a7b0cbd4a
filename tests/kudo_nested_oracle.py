"""CPU restatement of the reference's Kudo wire format for NESTED tables (LIST / STRUCT columns) -- TEST INFRASTRUCTURE
ONLY.  The flat restatement lives in oracle/kudo.py; this module generalises its writer and reader to column trees and
gives the same bytes for a flat table (tests/test_oracle_kudo_nested.py checks both).

Follows (file:line in /root/reference/src/main/java/com/nvidia/spark/rapids/jni/kudo/):
  KudoTableHeaderCalc.java:77-195, SlicedBufferSerializer.java:72-247 (writer), KudoTableMerger.java:96-295 (reader), in
  the visitor order of schema/HostColumnsVisitor.java.  The columns are flattened in pre-order (a LIST / STRUCT before
  its children) and the header's column count and hasValidity bits index that flattened list.  Every flattened column
  has a slice (offset, rows): the root slice is the header's, a STRUCT's children share their parent's slice, a LIST's
  child slice is (off[s], off[s + n] - off[s]) of the list's raw offsets.  Validity: STRUCT, LIST and leaf columns in
  pre-order (mask bytes of the slice, iff the column has a mask and the slice has rows); offsets: LIST offsets (n + 1
  raw int32 when n > 0) and STRING offsets in pre-order; data: leaves only.  Header, padding and the validity slice
  bytes are those of the flat format (oracle/kudo.py).
Pinned by the known answer of KudoSerializerTest.java:107-133 (buildSimpleTable, 172 bytes) and the merge known
answers of tests/test_oracle_kudo_nested.py.
"""
import struct
from typing import List, Sequence, Tuple

import numpy as np

from oracle import oracle as O
from oracle.kudo import MAGIC, _pad4, header_size  # noqa: F401  (the header and padding of the flat format)


def _visit(col: O.HCol, off: int, n: int, bitset: bytearray, idx: List[int], validity: bytearray, offsets: bytearray,
           data: bytearray) -> None:
    """One column of a partition and, depth first, its children: the slice is rows [off, off + n) of `col`."""
    c = idx[0]
    idx[0] += 1
    if col.mask is not None and n > 0:
        bitset[c // 8] |= 1 << (c % 8)
        b0 = off // 8
        validity += col.mask.view(np.uint8)[b0:(off + n - 1) // 8 + 1].tobytes()
    if col.type_id == O.STRUCT:
        for k in col.children or []:
            _visit(k, off, n, bitset, idx, validity, offsets, data)
    elif col.type_id == O.LIST:
        if n > 0:
            offsets += col.offsets[off:off + n + 1].astype("<i4").tobytes()
        s, e = (int(col.offsets[off]), int(col.offsets[off + n])) if col.offsets is not None and len(col.offsets) else (0, 0)
        _visit(col.children[0], s, e - s, bitset, idx, validity, offsets, data)
    elif col.type_id == O.STRING:
        if n > 0:
            offsets += col.offsets[off:off + n + 1].astype("<i4").tobytes()
            data += col.data[col.offsets[off]:col.offsets[off + n]].tobytes()
    else:
        sz = O.size_of(col.type_id)
        data += np.ascontiguousarray(col.data).view(np.uint8)[off * sz:(off + n) * sz].tobytes()


def num_flat(col: O.HCol) -> int:
    return 1 + sum(num_flat(k) for k in (col.children or []))


def flatten(cols: Sequence[O.HCol]) -> Tuple[List[int], List[int], List[int]]:
    """The pre-order schema of a table, as Schema.getFlattenedTypeIds / NumChildren / TypeScales give it."""
    ids, nch, scales = [], [], []

    def go(c):
        ids.append(c.type_id)
        nch.append(len(c.children or []) if c.type_id in (O.LIST, O.STRUCT) else 0)
        scales.append(c.scale)
        if c.type_id in (O.LIST, O.STRUCT):
            for k in c.children or []:
                go(k)
    for c in cols:
        go(c)
    return ids, nch, scales


def write_partition(cols: Sequence[O.HCol], row_offset: int, num_rows: int) -> bytes:
    nc = sum(num_flat(c) for c in cols)
    hs = header_size(nc)
    bitset = bytearray((nc + 7) // 8)
    validity, offsets, data = bytearray(), bytearray(), bytearray()
    idx = [0]
    for col in cols:
        _visit(col, row_offset, num_rows, bitset, idx, validity, offsets, data)
    vlen = _pad4(len(validity) + hs) - hs
    olen = _pad4(len(offsets))
    dlen = _pad4(len(data))
    head = struct.pack(">7i", MAGIC, row_offset, num_rows, vlen, olen, vlen + olen + dlen, nc) + bytes(bitset)
    return head + bytes(validity) + bytes(vlen - len(validity)) + bytes(offsets) + bytes(olen - len(offsets)) + bytes(data) + bytes(dlen - len(data))


def split(cols: Sequence[O.HCol], splits: Sequence[int]) -> Tuple[np.ndarray, np.ndarray]:
    """shuffle_split: `splits` = P + 1 row indices (0 ... n).  -> (uint8 buffer, int64 offsets[P + 1])."""
    parts = [write_partition(cols, int(splits[p]), int(splits[p + 1] - splits[p])) for p in range(len(splits) - 1)]
    offs = np.zeros(len(parts) + 1, dtype=np.int64)
    np.cumsum([len(p) for p in parts], out=offs[1:])
    return np.frombuffer(b"".join(parts), dtype=np.uint8).copy(), offs


class _Reader:
    """The sections of one partition, consumed in order."""

    def __init__(self, raw: bytes, base: int, nc: int):
        magic, self.roff, self.n, vlen, olen, total, ncols = struct.unpack(">7i", raw[base:base + 28])
        assert magic == MAGIC and ncols == nc, "not a Kudo header of this schema"
        hs = header_size(nc)
        self.raw, self.bitset = raw, raw[base + 28:base + hs]
        self.v, self.o, self.d = base + hs, base + hs + vlen, base + hs + vlen + olen

    def valid(self, c: int, off: int, n: int) -> np.ndarray:
        if (self.bitset[c // 8] >> (c % 8)) & 1 and n > 0:
            blen = (off + n - 1) // 8 - off // 8 + 1
            bits = np.unpackbits(np.frombuffer(self.raw[self.v:self.v + blen], dtype=np.uint8), bitorder="little")
            self.v += blen
            return bits[off % 8: off % 8 + n].astype(bool)
        return np.ones(n, dtype=bool)

    def offsets(self, n: int) -> np.ndarray:
        if n == 0:
            return np.zeros(1, np.int32)
        o = np.frombuffer(self.raw[self.o:self.o + 4 * (n + 1)], dtype="<i4").astype(np.int64)
        self.o += 4 * (n + 1)
        assert 0 <= o[0] <= o[-1], "decreasing offsets"
        return o

    def data(self, nbytes: int) -> bytes:
        b = self.raw[self.d:self.d + nbytes]
        self.d += nbytes
        return b


def _schema_tree(type_ids: Sequence[int], num_children: Sequence[int], scales: Sequence[int]):
    """Flattened pre-order schema -> list of (type_id, scale, [children]) roots."""
    pos = [0]

    def node():
        i = pos[0]
        pos[0] += 1
        t, k = int(type_ids[i]), int(num_children[i])
        assert t != O.LIST or k == 1, "a LIST has exactly one child"
        return (t, int(scales[i]), [node() for _ in range(k)], i)
    roots = []
    while pos[0] < len(type_ids):
        roots.append(node())
    return roots


def assemble_nested(buf: np.ndarray, part_offsets: np.ndarray, type_ids: Sequence[int], num_children: Sequence[int],
                    scales: Sequence[int] = None) -> List[O.HCol]:
    """shuffle_assemble / KudoTableMerger over a flattened schema: the partitions concatenated into one table."""
    nc = len(type_ids)
    roots = _schema_tree(type_ids, num_children, scales if scales is not None else [0] * nc)
    raw = buf.tobytes()
    # per flattened column: validity pieces, and offsets / bytes pieces (rebased when the column is built)
    valid = [[] for _ in range(nc)]
    offs = [[] for _ in range(nc)]          # LIST / STRING: per partition the n lengths
    data = [[] for _ in range(nc)]

    def read(node, r: _Reader, off: int, n: int):
        t, _, kids, c = node
        valid[c].append(r.valid(c, off, n))
        if t == O.STRUCT:
            for k in kids:
                read(k, r, off, n)
        elif t == O.LIST:
            o = r.offsets(n)
            offs[c].append(np.diff(o))
            read(kids[0], r, int(o[0]), int(o[-1] - o[0]))
        elif t == O.STRING:
            o = r.offsets(n)
            offs[c].append(np.diff(o))
            data[c].append(r.data(int(o[-1] - o[0])))
        else:
            data[c].append(r.data(n * O.size_of(t)))

    for p in range(len(part_offsets) - 1):
        r = _Reader(raw, int(part_offsets[p]), nc)
        for root in roots:
            read(root, r, r.roff, r.n)

    def build(node) -> O.HCol:
        t, scale, kids, c = node
        v = np.concatenate(valid[c]) if valid[c] else np.zeros(0, bool)
        mask = None if v.all() else O.pack_mask(v)
        if t in (O.LIST, O.STRING):
            lens = np.concatenate(offs[c]) if offs[c] else np.zeros(0, np.int64)
            o = np.zeros(len(v) + 1, dtype=np.int32)
            np.cumsum(lens, out=o[1:])
            if t == O.LIST:
                return O.HCol(O.LIST, None, mask, o, scale, len(v), [build(kids[0])])
            return O.HCol(O.STRING, np.frombuffer(b"".join(data[c]), dtype=np.uint8).copy(), mask, o, scale, len(v))
        if t == O.STRUCT:
            return O.HCol(O.STRUCT, None, mask, None, scale, len(v), [build(k) for k in kids])
        return O.HCol(t, np.frombuffer(b"".join(data[c]), dtype=np.uint8).copy(), mask, None, scale, len(v))
    return [build(r) for r in roots]


