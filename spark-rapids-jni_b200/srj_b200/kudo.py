"""The Kudo shuffle wire format on the device: host-side mirror of the reference's KudoGpuSerializer
(kudo/KudoGpuSerializer.java: splitAndSerializeToDevice / assembleFromDeviceRaw over shuffle_split / shuffle_assemble)
on the C ABI (include/srj_b200.h: srj_kudo_split_sizes / srj_kudo_split / srj_kudo_assemble_sizes / srj_kudo_assemble, and
srj_kudo_assemble_nested_sizes / srj_kudo_assemble_nested for schemas with LIST / STRUCT columns).

    buf, offsets = KudoGpuSerializer.splitAndSerializeToDevice(table, splits)   # splits: row indices 0 .. n (P + 1 of them)
    table = KudoGpuSerializer.assembleFromDeviceRaw(schema, buf, offsets)       # schema: a list of DTypes, or a Schema

Split writes flat tables; assemble reads flat and nested ones (a map is LIST<STRUCT<K, V>>).
"""
import ctypes as C
from typing import List, Sequence, Tuple

import numpy as np
import torch

from . import _native as N
from . import ColumnVector, DType, Schema, Table, _as_dtype, _carray, _empty, _stream_ptr


class KudoGpuSerializer:
    @staticmethod
    def splitAndSerializeToDevice(table: Table, splits) -> Tuple[torch.Tensor, torch.Tensor]:
        """-> (uint8 device buffer with the P partitions back to back, int64 device offsets[P + 1])."""
        cols = table.columns
        n = table.getRowCount()
        dev = next((t.device for c in cols for t in (c.data, c.offsets, c.mask) if t is not None), torch.device("cuda", torch.cuda.current_device()))
        lib = N.lib()
        with torch.cuda.device(dev):
            st = _stream_ptr()
            d_splits = splits if isinstance(splits, torch.Tensor) else torch.tensor(list(splits), dtype=torch.int32, device=dev)
            d_splits = d_splits.to(torch.int32)
            P = d_splits.numel() - 1
            ws = _empty(lib.srj_kudo_workspace_bytes(len(cols), P), torch.uint8, dev)
            offs = _empty(P + 1, torch.int64, dev)
            total = C.c_int64(0)
            carr = _carray(cols)
            N.check(lib.srj_kudo_split_sizes(carr, len(cols), n, d_splits.data_ptr(), P, offs.data_ptr(), C.byref(total), ws.data_ptr(), st),
                    "kudo split")
            buf = _empty(total.value, torch.uint8, dev)
            N.check(lib.srj_kudo_split(carr, len(cols), n, d_splits.data_ptr(), P, offs.data_ptr(), buf.data_ptr(), ws.data_ptr(), st), "kudo split")
        return buf, offs

    @staticmethod
    def assembleFromDeviceRaw(schema, buf: torch.Tensor, offsets: torch.Tensor) -> Table:
        """The partitions (device buffer + int64 offsets[P + 1]) concatenated into one table.  `schema`: a Schema (LIST
        columns come back with `child`, STRUCT columns with `children`), or a sequence of DTypes of a flat table."""
        if isinstance(schema, Schema):
            return KudoGpuSerializer._assemble_nested(schema, buf, offsets)
        dts = [_as_dtype(d) for d in schema]
        dev = buf.device
        lib = N.lib()
        P = offsets.numel() - 1
        with torch.cuda.device(dev):
            st = _stream_ptr()
            ws = _empty(lib.srj_kudo_workspace_bytes(len(dts), P), torch.uint8, dev)
            ids = (C.c_int32 * len(dts))(*[d.type_id for d in dts])
            rows = C.c_int64(0)
            chars = (C.c_int64 * len(dts))()
            N.check(lib.srj_kudo_assemble_sizes(buf.data_ptr(), offsets.data_ptr(), P, ids, len(dts), C.byref(rows), chars, ws.data_ptr(), st),
                    "kudo assemble")
            n = rows.value
            words = (n + 31) // 32
            outs: List[ColumnVector] = []
            for i, d in enumerate(dts):
                mask = _empty(max(1, words), torch.int32, dev)
                if d.type_id == DType.STRING:
                    outs.append(ColumnVector(d, n, _empty(int(chars[i]), torch.uint8, dev), mask, _empty(n + 1, torch.int32, dev)))
                else:
                    outs.append(ColumnVector(d, n, _empty(n * d.size_in_bytes(), torch.uint8, dev), mask))
            N.check(lib.srj_kudo_assemble(buf.data_ptr(), offsets.data_ptr(), P, _carray(outs), len(dts), n, ws.data_ptr(), st), "kudo assemble")
        return Table(outs)

    @staticmethod
    def _assemble_nested(schema: Schema, buf: torch.Tensor, offsets: torch.Tensor) -> Table:
        ids, nch, scales = schema.getFlattenedTypeIds(), schema.getFlattenedNumChildren(), schema.getFlattenedTypeScales()
        F = len(ids)
        dev = buf.device
        lib = N.lib()
        P = offsets.numel() - 1
        with torch.cuda.device(dev):
            st = _stream_ptr()
            ws = _empty(lib.srj_kudo_nested_workspace_bytes(F, P), torch.uint8, dev)
            rows = (C.c_int64 * max(F, 1))()
            chars = (C.c_int64 * max(F, 1))()
            N.check(lib.srj_kudo_assemble_nested_sizes(buf.data_ptr(), offsets.data_ptr(), P, (C.c_int32 * max(F, 1))(*ids),
                                                       (C.c_int32 * max(F, 1))(*nch), F, rows, chars, ws.data_ptr(), st), "kudo assemble")
            pos = [0]

            def build() -> ColumnVector:       # the flattened columns back into trees, in pre-order
                c = pos[0]
                pos[0] += 1
                d, n = DType(ids[c], scales[c]), int(rows[c])
                mask = _empty(max(1, (n + 31) // 32), torch.int32, dev)
                if d.type_id == DType.LIST:
                    offs = _empty(n + 1, torch.int32, dev)
                    return ColumnVector(d, n, None, mask, offs, build())
                if d.type_id == DType.STRUCT:
                    return ColumnVector(d, n, None, mask, children=[build() for _ in range(nch[c])])
                if d.type_id == DType.STRING:
                    return ColumnVector(d, n, _empty(int(chars[c]), torch.uint8, dev), mask, _empty(n + 1, torch.int32, dev))
                return ColumnVector(d, n, _empty(n * d.size_in_bytes(), torch.uint8, dev), mask)
            outs: List[ColumnVector] = []
            while pos[0] < F:
                outs.append(build())
            N.check(lib.srj_kudo_assemble_nested(buf.data_ptr(), offsets.data_ptr(), P, _carray(outs), len(outs), ws.data_ptr(), st),
                    "kudo assemble")
        return Table(outs)
