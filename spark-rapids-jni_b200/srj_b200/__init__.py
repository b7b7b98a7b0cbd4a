"""srj_b200 -- host-side mirror of the reference's Java surface for the row<->columnar + hash path.

The reference host code is Java (`com.nvidia.spark.rapids.jni.RowConversion` / `Hash` over
`ai.rapids.cudf.{Table,ColumnVector,ColumnView,DType}`); no JDK exists in this image, so the same
surface -- same class and method names, argument meaning and error behaviour -- is mirrored here in
Python over torch device tensors, calling the C ABI of libsrj_b200.so exactly as the JNI shim
would (INTEGRATION.md).  torch is used for device memory and streams only.

  RowConversion.convertToRows(table)                      RowConversion.java:35-42
  RowConversion.convertToRowsFixedWidthOptimized(table)   RowConversion.java:118-125
  RowConversion.convertFromRows(vec, *schema)             RowConversion.java:137-146
  RowConversion.convertFromRowsFixedWidthOptimized(...)   RowConversion.java:158-167
  Hash.murmurHash32(seed, columns) / Hash.murmurHash32(columns)   Hash.java:34-62
  Hash.xxhash64(seed, columns) / Hash.xxhash64(columns)           Hash.java:64-89
  Hash.hiveHash(columns)                                           Hash.java:91-105
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _native as N
from ._native import CudfColumnSizeOverflowException, CudfException, CudaException  # noqa: F401

__all__ = ["DType", "Schema", "ColumnVector", "ColumnView", "Table", "RowConversion", "Hash", "CudfException",
           "CudfColumnSizeOverflowException", "Plan"]


class DType:
    """ai.rapids.cudf.DType: native type id + scale (dtype_utils.hpp:44-54)."""
    (EMPTY, INT8, INT16, INT32, INT64, UINT8, UINT16, UINT32, UINT64, FLOAT32, FLOAT64, BOOL8,
     TIMESTAMP_DAYS, TIMESTAMP_SECONDS, TIMESTAMP_MILLISECONDS, TIMESTAMP_MICROSECONDS, TIMESTAMP_NANOSECONDS,
     DURATION_DAYS, DURATION_SECONDS, DURATION_MILLISECONDS, DURATION_MICROSECONDS, DURATION_NANOSECONDS,
     DICTIONARY32, STRING, LIST, DECIMAL32, DECIMAL64, DECIMAL128, STRUCT) = range(29)

    _SIZES = {1: (1, 5, 11), 2: (2, 6), 4: (3, 7, 9, 12, 17, 25), 8: (4, 8, 10, 13, 14, 15, 16, 18, 19, 20, 21, 26),
              16: (27,)}

    def __init__(self, type_id: int, scale: int = 0):
        self.type_id = int(type_id)
        self.scale = int(scale)

    @staticmethod
    def create(type_id: int, scale: int = 0) -> "DType":
        return DType(type_id, scale)

    def size_in_bytes(self) -> int:
        for sz, ids in DType._SIZES.items():
            if self.type_id in ids:
                return sz
        return 0

    def is_fixed_width(self) -> bool:
        return self.size_in_bytes() > 0

    def __eq__(self, o):
        return isinstance(o, DType) and (self.type_id, self.scale) == (o.type_id, o.scale)

    def __repr__(self):
        return f"DType({self.type_id}, scale={self.scale})"


class Schema:
    """ai.rapids.cudf.Schema: the column types of a table as a tree (LIST / STRUCT columns have children), and its
    pre-order flattening -- the form the Kudo reader takes (KudoGpuSerializer.assembleFromDeviceRaw).

        b = Schema.builder()
        b.column(DType(DType.INT64), "key")
        lst = b.addColumn(DType(DType.LIST), "xs"); lst.column(DType(DType.INT32), "x")
        schema = b.build()
    """

    class Builder:
        def __init__(self, dtype: Optional["DType"] = None, name: Optional[str] = None):
            self.dtype, self.name = dtype, name
            self.children: List["Schema.Builder"] = []

        def addColumn(self, dtype, name: str) -> "Schema.Builder":
            """Add a column; for LIST and STRUCT the returned builder takes its children, otherwise this builder."""
            child = Schema.Builder(_as_dtype(dtype), name)
            self.children.append(child)
            return child if child.dtype.type_id in (DType.LIST, DType.STRUCT) else self

        def column(self, dtype, name: str) -> "Schema.Builder":
            self.addColumn(dtype, name)
            return self

        def build(self) -> "Schema":
            return Schema(self)

    def __init__(self, root: "Schema.Builder"):
        self._root = root

    @staticmethod
    def builder() -> "Schema.Builder":
        return Schema.Builder()

    def _flat(self) -> List["Schema.Builder"]:
        out: List[Schema.Builder] = []

        def go(b):
            out.append(b)
            for k in b.children:
                go(k)
        for k in self._root.children:
            go(k)
        return out

    def getColumnNames(self) -> List[str]:
        return [k.name for k in self._root.children]

    def getNumChildren(self) -> int:
        return len(self._root.children)

    def getFlattenedNumColumns(self) -> int:
        return len(self._flat())

    def getFlattenedTypeIds(self) -> List[int]:
        return [b.dtype.type_id for b in self._flat()]

    def getFlattenedNumChildren(self) -> List[int]:
        return [len(b.children) for b in self._flat()]

    def getFlattenedTypeScales(self) -> List[int]:
        return [b.dtype.scale for b in self._flat()]


def _as_dtype(d) -> DType:
    return d if isinstance(d, DType) else DType(int(d))


def _stream_ptr() -> int:
    return int(torch.cuda.current_stream().cuda_stream)


class ColumnView:
    """The cudf::column_view fields this path uses, held as torch CUDA tensors.

    fixed width : data = uint8 tensor [size * size_of(type)]
    STRING      : data = uint8 chars, offsets = int32 [size + 1]
    LIST<INT8>  : offsets = int32 [size + 1], child = ColumnView(INT8 bytes)   (the rows column)
    mask        : int32 tensor of ceil(size/32) words or None (= all valid)
    """

    def __init__(self, dtype, size: int, data: Optional[torch.Tensor] = None, mask: Optional[torch.Tensor] = None,
                 offsets: Optional[torch.Tensor] = None, child: Optional["ColumnView"] = None,
                 null_count: Optional[int] = None, children: Optional[Sequence["ColumnView"]] = None):
        self.dtype = _as_dtype(dtype)
        self.size = int(size)
        self.data = data
        self.mask = mask
        self.offsets = offsets
        self.child = child                 # LIST: the element column
        self.children = list(children) if children is not None else None   # STRUCT: the fields
        self._null_count = null_count

    @staticmethod
    def makeStructView(*fields: "ColumnView", mask: Optional[torch.Tensor] = None) -> "ColumnView":
        """ai.rapids.cudf.ColumnView.makeStructView: a STRUCT view over existing columns (all the same row count)."""
        n = fields[0].size if fields else 0
        return ColumnView(DType.STRUCT, n, None, mask, None, None, None, children=fields)

    @staticmethod
    def makeListView(offsets: torch.Tensor, child: "ColumnView", mask: Optional[torch.Tensor] = None) -> "ColumnView":
        """A LIST view: int32 offsets[rows + 1] into `child`."""
        return ColumnView(DType.LIST, offsets.numel() - 1, None, mask, offsets, child)

    # --- ai.rapids.cudf.ColumnView-ish accessors
    def getRowCount(self) -> int:
        return self.size

    def getType(self) -> DType:
        return self.dtype

    def getNullCount(self) -> int:
        if self._null_count is None:
            if self.mask is None:
                self._null_count = 0
            else:
                self._null_count = self.size - int(np.unpackbits(
                    self.mask.cpu().numpy().view(np.uint8), bitorder="little")[: self.size].sum())
        return self._null_count

    def close(self):
        self.data = self.mask = self.offsets = self.child = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # --- construction / extraction helpers (test + bench plumbing)
    @staticmethod
    def from_numpy(type_id: int, data: Optional[np.ndarray], mask: Optional[np.ndarray] = None,
                   offsets: Optional[np.ndarray] = None, scale: int = 0, size: Optional[int] = None,
                   device="cuda") -> "ColumnVector":
        dt = DType(type_id, scale)

        def up(a, npdt):
            if a is None:
                return None
            a = np.ascontiguousarray(a)
            t = torch.from_numpy(a.view(npdt).copy() if a.size else np.zeros(0, npdt))
            return t.to(device)
        d = up(data.view(np.uint8) if data is not None else None, np.uint8)
        m = up(mask.view(np.int32) if mask is not None else None, np.int32)
        o = up(offsets.view(np.int32) if offsets is not None else None, np.int32)
        if size is None:
            size = (len(offsets) - 1) if type_id == DType.STRING else (data.nbytes // max(1, dt.size_in_bytes()))
        return ColumnVector(dt, size, d, m, o)

    def to_numpy(self):
        """-> (data uint8 ndarray | None, mask uint32 ndarray | None, offsets int32 ndarray | None)"""
        d = self.data.cpu().numpy().view(np.uint8) if self.data is not None else None
        m = self.mask.cpu().numpy().view(np.uint32) if self.mask is not None else None
        o = self.offsets.cpu().numpy() if self.offsets is not None else None
        return d, m, o

    def _c(self) -> N.SrjColumn:
        c = N.SrjColumn()
        c.type_id = self.dtype.type_id
        c.scale = self.dtype.scale
        c.size = self.size
        c.data = self.data.data_ptr() if self.data is not None and self.data.numel() else None
        c.null_mask = self.mask.data_ptr() if self.mask is not None else None
        c.offsets = self.offsets.data_ptr() if self.offsets is not None else None
        kids = None
        if self.dtype.type_id == DType.LIST and self.child is not None:
            kids = [self.child]
        elif self.dtype.type_id == DType.STRUCT and self.children:
            kids = self.children
        if kids:
            arr = (N.SrjColumn * len(kids))()
            for i, k in enumerate(kids):
                arr[i] = k._c()
            c.children = arr
            c.num_children = len(kids)
            self._c_keep = arr           # the child descriptors must outlive the call (the view does)
        return c


class ColumnVector(ColumnView):
    """Owning column (ai.rapids.cudf.ColumnVector): same fields, owns its tensors."""


class Table:
    """ai.rapids.cudf.Table: an ordered set of equal-length columns."""

    def __init__(self, *columns: ColumnView):
        if len(columns) == 1 and isinstance(columns[0], (list, tuple)):
            columns = tuple(columns[0])
        self.columns: List[ColumnView] = list(columns)
        rows = {c.size for c in self.columns}
        if len(rows) > 1:
            raise ValueError("All columns must have the same number of rows")
        self.rows = rows.pop() if rows else 0

    def getNumberOfColumns(self) -> int:
        return len(self.columns)

    def getRowCount(self) -> int:
        return self.rows

    def getColumn(self, i: int) -> ColumnView:
        return self.columns[i]

    def close(self):
        for c in self.columns:
            c.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


def _carray(cols: Sequence[ColumnView]):
    arr = (N.SrjColumn * max(1, len(cols)))()
    for i, c in enumerate(cols):
        arr[i] = c._c()
    return arr


class Plan:
    """Schema-keyed cache of srj_plan handles (what the JNI shim keeps per schema)."""
    _cache = {}

    def __init__(self, dtypes: Sequence[DType]):
        self.dtypes = [_as_dtype(d) for d in dtypes]
        n = len(self.dtypes)
        t = np.array([d.type_id for d in self.dtypes], dtype=np.int32)
        s = np.array([d.scale for d in self.dtypes], dtype=np.int32)
        h = C.c_void_p()
        N.check(N.lib().srj_plan_create(t.ctypes.data_as(C.c_void_p) if n else None,
                                        s.ctypes.data_as(C.c_void_p) if n else None, n, C.byref(h)), "plan_create")
        self.handle = h
        lay = N.SrjLayout()
        N.check(N.lib().srj_plan_layout(self.handle, C.byref(lay)))
        self.layout = lay

    @staticmethod
    def get(dtypes: Sequence[DType]) -> "Plan":
        key = (torch.cuda.current_device(), tuple((d.type_id, d.scale) for d in map(_as_dtype, dtypes)))
        p = Plan._cache.get(key)
        if p is None:
            p = Plan._cache[key] = Plan(dtypes)
        return p

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                N.lib().srj_plan_destroy(self.handle)
        except Exception:
            pass


def _empty(n, dtype, device):
    return torch.empty(int(n), dtype=dtype, device=device)


class RowConversion:
    """com.nvidia.spark.rapids.jni.RowConversion (RowConversion.java:22-174)."""
    MAX_BATCHES = 4096

    @staticmethod
    def convertToRows(table: Table) -> List[ColumnVector]:
        """Table -> one LIST<INT8> ColumnVector per <= 2 GiB batch (RowConversion.java:35-42, RC:1994-2055)."""
        if table is None:
            raise TypeError("input table is null")           # JNI_NULL_CHECK, RowConversionJni.cpp:49
        cols = table.columns
        if not cols:
            raise CudfException("convert_to_rows: a table needs at least one column")
        dev = cols[0].data.device if cols[0].data is not None else cols[0].offsets.device
        with torch.cuda.device(dev):
            plan = Plan.get([c.dtype for c in cols])
            n = table.getRowCount()
            lib = N.lib()
            carr = _carray(cols)
            stream = _stream_ptr()
            ws_bytes = lib.srj_to_rows_workspace_bytes(plan.handle, n)
            ws = _empty(max(ws_bytes, 8), torch.uint8, dev)
            batches = (N.SrjRowBatch * RowConversion.MAX_BATCHES)()
            nb = C.c_int32(0)
            N.check(lib.srj_to_rows_plan_batches(plan.handle, carr, n, ws.data_ptr(), batches,
                                                 RowConversion.MAX_BATCHES, C.byref(nb), stream), "convertToRows")
            if nb.value == 0:
                # empty table: one empty LIST column (the reference reads row_batches[0] of an empty
                # vector here, SURVEY App. C.4)
                off = torch.zeros(1, dtype=torch.int32, device=dev)
                return [ColumnVector(DType.LIST, 0, None, None, off,
                                     ColumnVector(DType.INT8, 0, _empty(0, torch.uint8, dev)))]
            outs, optrs, dptrs = [], (C.c_void_p * nb.value)(), (C.c_void_p * nb.value)()
            for b in range(nb.value):
                off = _empty(batches[b].row_count + 1, torch.int32, dev)
                dat = _empty(batches[b].num_bytes, torch.uint8, dev)
                optrs[b], dptrs[b] = off.data_ptr(), dat.data_ptr()
                outs.append(ColumnVector(DType.LIST, batches[b].row_count, None, None, off,
                                         ColumnVector(DType.INT8, batches[b].num_bytes, dat), null_count=0))
            N.check(lib.srj_convert_to_rows(plan.handle, carr, n, ws.data_ptr(), batches, nb.value, optrs, dptrs,
                                            stream), "convertToRows")
            return outs

    @staticmethod
    def convertToRowsFixedWidthOptimized(table: Table) -> List[ColumnVector]:
        """Legacy entry point (RowConversion.java:118-125, RC:2057-2125): fixed-width tables only, same row
        bytes as convertToRows; both map onto one kernel family here."""
        for c in table.columns:
            if not c.dtype.is_fixed_width():
                raise CudfException("Only fixed width types are currently supported")   # RC:2122-2124
        plan = Plan.get([c.dtype for c in table.columns])
        if plan.layout.fixed_row_size * 32 > 48 * 1024:                                # RC:1184-1191
            raise CudfException("Row size is too large to fit in shared memory")
        return RowConversion.convertToRows(table)

    @staticmethod
    def convertFromRows(vec: ColumnView, *schema) -> Table:
        """LIST<INT8> rows + schema -> Table (RowConversion.java:137-146, RC:2149-2441)."""
        return RowConversion._from_rows(vec, schema, None)

    @staticmethod
    def _from_rows(vec: ColumnView, schema, fused):
        if vec is None:
            raise TypeError("input column is null")
        if len(schema) == 1 and isinstance(schema[0], (list, tuple)):
            schema = tuple(schema[0])
        dts = [_as_dtype(d) for d in schema]
        if vec.dtype.type_id != DType.LIST or vec.child is None or vec.child.dtype.type_id not in (DType.INT8,
                                                                                                   DType.UINT8):
            raise CudfException("Only a list of bytes is supported as input")          # RC:2157-2158
        child = vec.child
        dev = vec.offsets.device
        with torch.cuda.device(dev):
            plan = Plan.get(dts)
            n = vec.size
            lib = N.lib()
            stream = _stream_ptr()
            words = (n + 31) // 32
            outs: List[ColumnVector] = []
            for d in dts:
                mask = _empty(words, torch.int32, dev)                                 # always allocated, RC:2220
                if d.type_id == DType.STRING:
                    outs.append(ColumnVector(d, n, None, mask, _empty(n + 1, torch.int32, dev)))
                else:
                    outs.append(ColumnVector(d, n, _empty(n * d.size_in_bytes(), torch.uint8, dev), mask))
            nc = len(dts)
            nulls = torch.zeros(max(nc, 1), dtype=torch.int64, device=dev)
            totals = torch.zeros(nc + 1, dtype=torch.int64, device=dev)   # + status word for phase 2
            carr = _carray(outs)
            rows_ptr = child.data.data_ptr() if child.data is not None and child.data.numel() else None
            ws_bytes = lib.srj_from_rows_workspace_bytes(plan.handle, n)
            ws = _empty(ws_bytes, torch.uint8, dev) if ws_bytes else None          # rmm allocation in the JNI shim
            ws_ptr = ws.data_ptr() if ws is not None else None
            fh, hout = None, None
            if fused is not None:
                key_columns, kind, seed = fused
                fh = N.SrjFusedHash()
                fh.kind = {"xxhash64": N.HASH_XXHASH64, "murmur3": N.HASH_MURMUR3_32, "hive": N.HASH_HIVE}[kind]
                fh.num_keys = len(key_columns)
                for i, k in enumerate(key_columns):
                    fh.key_columns[i] = int(k)
                fh.seed = int(seed)
                hout = _empty(n, torch.int64 if kind == "xxhash64" else torch.int32, dev)
                fh.out = hout.data_ptr()
            N.check(lib.srj_convert_from_rows_fixed(plan.handle, rows_ptr, vec.offsets.data_ptr(), child.size, n,
                                                    carr, nulls.data_ptr(), totals.data_ptr(),
                                                    C.byref(fh) if fh is not None else None, ws_ptr, stream),
                    "convertFromRows")
            if plan.layout.num_string_columns:
                h_tot = totals.cpu().numpy()                                           # the sync of RC:2389
                for i, d in enumerate(dts):
                    if d.type_id == DType.STRING:
                        if h_tot[i] > 2**31 - 1 or (int(h_tot[nc]) & 2):
                            raise CudfColumnSizeOverflowException(f"string column {i} exceeds the int32 chars limit")
                        outs[i].data = _empty(int(h_tot[i]), torch.uint8, dev)
                carr = _carray(outs)
                N.check(lib.srj_convert_from_rows_strings(plan.handle, rows_ptr, vec.offsets.data_ptr(), child.size, n,
                                                          carr, totals.data_ptr(), ws_ptr, stream), "convertFromRows")
            h_nulls = nulls.cpu().numpy()
            for i, o in enumerate(outs):
                o._null_count = int(h_nulls[i])
            if fused is not None:
                kind = fused[1]
                return Table(outs), ColumnVector(DType.INT64 if kind == "xxhash64" else DType.INT32, n,
                                                 hout.view(torch.uint8), None, null_count=0)
            return Table(outs)

    @staticmethod
    def convertFromRowsFixedWidthOptimized(vec: ColumnView, *schema) -> Table:
        """Legacy entry point (RowConversion.java:158-167, RC:2443-2512)."""
        if len(schema) == 1 and isinstance(schema[0], (list, tuple)):
            schema = tuple(schema[0])
        dts = [_as_dtype(d) for d in schema]
        for d in dts:
            if not d.is_fixed_width():
                raise CudfException("Only fixed width types are currently supported")   # RC:2509-2511
        plan = Plan.get(dts)
        if vec.child is not None and plan.layout.fixed_row_size * vec.size != vec.child.size:
            raise CudfException("The layout of the data appears to be off")            # RC:2465
        return RowConversion.convertFromRows(vec, *dts)

    # fused from_rows + partition hash (BASELINE config 4); not in the Java surface, used by the plugin-side
    # GpuHashPartitioning equivalent and by bench.py.  Keys are fixed-width columns; the schema may hold STRING columns.
    @staticmethod
    def convertFromRowsWithHash(vec: ColumnView, schema, key_columns: Sequence[int], kind: str = "xxhash64",
                                seed: int = 42):
        dts = [_as_dtype(d) for d in schema]
        for k in key_columns:
            if not dts[int(k)].is_fixed_width():
                raise CudfException("fused hash path: keys must be fixed-width columns")
        return RowConversion._from_rows(vec, dts, (list(key_columns), kind, seed))


class Hash:
    """com.nvidia.spark.rapids.jni.Hash (Hash.java:26-105)."""
    DEFAULT_XXHASH64_SEED = 42
    MAX_STACK_DEPTH = 8

    @staticmethod
    def getMaxStackDepth() -> int:
        return N.lib().srj_get_max_stack_depth()

    @staticmethod
    def _prep(columns):
        cols = list(columns)
        if not cols:
            raise AssertionError("expected at least one column")            # Hash.java:47
        n = cols[0].size
        for c in cols:
            assert c is not None, "Column vectors passed may not be null"
            assert c.size == n, "Row count mismatch, all columns must be the same size"   # Hash.java:51-53
            assert not (17 <= c.dtype.type_id <= 21), "Unsupported column type Duration"  # Hash.java:54
        def device_of(c):
            for t in (c.data, c.offsets, c.mask):
                if t is not None:
                    return t.device
            for k in ([c.child] if c.child is not None else []) + list(c.children or []):
                d = device_of(k)
                if d is not None:
                    return d
            return None
        dev = next((d for d in map(device_of, cols) if d is not None), torch.device("cuda", torch.cuda.current_device()))
        return cols, n, dev

    @staticmethod
    def murmurHash32(*args) -> ColumnVector:
        """murmurHash32(seed, columns) or murmurHash32(columns) (seed 0) -> INT32 column."""
        seed, columns = (args[0], args[1]) if len(args) == 2 else (0, args[0])
        cols, n, dev = Hash._prep(columns)
        with torch.cuda.device(dev):
            out = _empty(n, torch.int32, dev)
            N.check(N.lib().srj_murmur_hash3_32(_carray(cols), len(cols), n, C.c_uint32(seed & 0xFFFFFFFF),
                                                out.data_ptr(), _stream_ptr()), "murmurHash32")
            return ColumnVector(DType.INT32, n, out.view(torch.uint8), None, null_count=0)

    @staticmethod
    def xxhash64(*args) -> ColumnVector:
        """xxhash64(seed, columns) or xxhash64(columns) (seed 42) -> INT64 column."""
        seed, columns = (args[0], args[1]) if len(args) == 2 else (Hash.DEFAULT_XXHASH64_SEED, args[0])
        cols, n, dev = Hash._prep(columns)
        with torch.cuda.device(dev):
            out = _empty(n, torch.int64, dev)
            N.check(N.lib().srj_xxhash64(_carray(cols), len(cols), n, C.c_int64(seed), out.data_ptr(),
                                         _stream_ptr()), "xxhash64")
            return ColumnVector(DType.INT64, n, out.view(torch.uint8), None, null_count=0)

    @staticmethod
    def hiveHash(columns) -> ColumnVector:
        cols, n, dev = Hash._prep(columns)
        with torch.cuda.device(dev):
            out = _empty(n, torch.int32, dev)
            N.check(N.lib().srj_hive_hash(_carray(cols), len(cols), n, out.data_ptr(), _stream_ptr()), "hiveHash")
            return ColumnVector(DType.INT32, n, out.view(torch.uint8), None, null_count=0)
