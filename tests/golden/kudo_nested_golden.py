"""Nested Kudo tables transcribed from the reference's own tests (src/test/java/com/nvidia/spark/rapids/jni/kudo/):
KudoSerializerTest.java -- buildSimpleTable (:339-353) with the known answer of testWriteSimple (:107-133),
buildEmptyStructTable (:355-373), buildTestTable (:375-512), the slicing loop of :56-71 and the merge known answers of
testMergeList (:201-236) and testMergeComplexStructList (:238-267); KudoGpuSerializerTest.java -- buildMediumTable
(:416-438), buildHalfEmptyStructTable (:451-465), buildStringListTable (:506-513) and calcEvenSlices (:217-231).

Columns are built the way cudf's Table.TestBuilder builds them: a column gets a validity mask only if it holds a null
(the 172-byte answer depends on it), a null STRUCT row is null in every field, a null LIST row has no elements.
Specs: a leaf type name, ("DEC32" | "DEC64" | "DEC128", scale), ("LIST", child) or ("STRUCT", [fields])."""
import numpy as np

from oracle import oracle as O

INT_MIN, INT_MAX = -2**31, 2**31 - 1
FLT_MAX, FLT_MIN = float(np.finfo(np.float32).max), 1.4e-45          # Float.MAX_VALUE, Float.MIN_VALUE (denormal)

_LEAF = {"INT8": O.INT8, "INT16": O.INT16, "INT32": O.INT32, "INT64": O.INT64, "FLOAT32": O.FLOAT32, "FLOAT64": O.FLOAT64,
         "BOOL8": O.BOOL8, "STRING": O.STRING, "TS_DAYS": O.TIMESTAMP_DAYS, "TS_MS": O.TIMESTAMP_MILLISECONDS,
         "TS_S": O.TIMESTAMP_SECONDS, "DEC32": O.DECIMAL32, "DEC64": O.DECIMAL64, "DEC128": O.DECIMAL128}
_NP = {O.INT8: np.int8, O.INT16: np.int16, O.INT32: np.int32, O.INT64: np.int64, O.FLOAT32: np.float32, O.FLOAT64: np.float64,
       O.BOOL8: np.uint8, O.TIMESTAMP_DAYS: np.int32, O.TIMESTAMP_MILLISECONDS: np.int64, O.TIMESTAMP_SECONDS: np.int64,
       O.DECIMAL32: np.int32, O.DECIMAL64: np.int64}


def _mask(valid):
    valid = np.asarray(valid, bool)
    return None if valid.all() else O.pack_mask(valid)


def col(spec, values) -> O.HCol:
    """A host column of `spec` from python values (None = null)."""
    n = len(values)
    valid = [v is not None for v in values]
    if isinstance(spec, tuple) and spec[0] == "LIST":
        offs, flat = [0], []
        for v in values:
            flat.extend(v or [])
            offs.append(len(flat))
        return O.HCol(O.LIST, None, _mask(valid), np.array(offs, np.int32), 0, n, [col(spec[1], flat)])
    if isinstance(spec, tuple) and spec[0] == "STRUCT":
        kids = [col(f, [None if v is None else v[i] for v in values]) for i, f in enumerate(spec[1])]
        return O.HCol(O.STRUCT, None, _mask(valid), None, 0, n, kids)
    name, scale = (spec, 0) if isinstance(spec, str) else spec
    t = _LEAF[name]
    if t == O.STRING:
        return O.strings_col([None if v is None else v.encode() for v in values])
    if t == O.DECIMAL128:
        data = b"".join(int(v or 0).to_bytes(16, "little", signed=True) for v in values)
        return O.HCol(t, np.frombuffer(data, np.uint8).copy(), _mask(valid), None, scale, n)
    data = np.array([0 if v is None else v for v in values], dtype=_NP[t])
    return O.HCol(t, data.view(np.uint8).copy(), _mask(valid), None, scale, n)


def table(*cols):
    return [col(s, v) for s, v in cols]


def slice_size_loop(n):
    """KudoSerializerTest.java:56-71: for every slice size n .. 1, the table cut into consecutive slices of that size."""
    return [list(range(0, n, size)) + [n] for size in range(n, 0, -1)]


def calc_even_slices(n, num_slices):
    """KudoGpuSerializerTest.java:217-231 (interior split points) as splits 0 .. n."""
    per = n // num_slices
    return [0] + [per * (i + 1) for i in range(num_slices - 1)] + [n]


def even_slicings(n):
    """KudoGpuSerializerTest's round trips: numSlices = 1 .. rows - 1."""
    return [calc_even_slices(n, k) for k in range(1, max(n, 2))]


# ---- KudoSerializerTest.java ------------------------------------------------------------------------------------------
def build_simple_table():           # :339-353
    st = ("STRUCT", ["INT8", "INT64"])
    return table(("INT32", [1, 2, 3, 4]),
                 ("STRING", ["1", "12", None, "45"]),
                 (("LIST", "INT32"), [[1, None, 3], [4, 5, 6], None, [7, 8, 9]]),
                 (st, [(1, 11), (2, None), None, (3, 33)]))


# testWriteSimple (:107-133): rows [0, 4) -> 172 bytes; header fields and hasValidity bits
SIMPLE_KNOWN = dict(bytes=172, num_columns=7, offset=0, num_rows=4, validity_len=7, offsets_len=40, total_len=143,
                    has_validity=[False, True, True, True, True, True, True])


def build_empty_struct_table():     # :355-373
    s, z = (), None
    vals = [s, z, z, s, z, z, s, s, z, s, s, z, s, s, z, z,
            s, z, z, s, z, z, s, s, z, s, s, z, s, s, z, z,
            s, s, z, s, z, z, s, s, z, s, s, z, s, z, z, z,
            s, z, z, s, z, s, s, z, z, s, s, z, s, s, z, z,
            s, z, z, s, z, z, s, s, z, s, s, z, s, s, z, z,
            s, z, z, z, z, z, s, s, z, s, s, z, s, s, z, z,
            s]
    return table((("STRUCT", []), vals))


def _kv(*pairs):
    return [None if p is None else tuple(p) for p in pairs]


def build_test_table():             # :375-512
    N = None
    list_map = ("LIST", ("LIST", ("STRUCT", ["STRING", "STRING"])))
    map_struct = ("LIST", ("STRUCT", ["STRING", "STRING"]))
    struct_t = ("STRUCT", ["INT32", "FLOAT32"])
    list_date = ("LIST", ("STRUCT", ["INT32", "INT32"]))
    odd_nulls = [100, 202, 3003, 40004, 5, -60, 1, N, 3, N, 5, N, 7, N, 9, N, 11, N, 13, N, 15]
    longs = [1, N, 1001, 50, -2000, N, 1, 2, 3, 4, N, 6, 7, 8, 9, N, 11, 12, 13, 14, N]
    null_lists = [[N] * 2, [N] * 4, [], [N] * 3, [], [N] * 5, [N], [N] * 3, [N] * 2, [N] * 4, [N] * 5, [], [N] * 4, [N] * 3,
                  [N] * 2, [N] * 3, [N] * 2, [N], [N], [N] * 2, [N] * 5]
    return table(
        ("INT32", odd_nulls),
        ("BOOL8", [1, 1, 0, 0, 1, N, 1, 1, N, 0, 0, N, 1, 1, N, 0, 0, N, 1, 1, N]),
        ("INT8", [1, 2, N, 4, 5, 6, 1, 2, 3, N, 5, 6, 7, N, 9, 10, 11, N, 13, 14, 15]),
        ("INT16", [6, 5, 4, N, 2, 1, 1, 2, 3, N, 5, 6, 7, N, 9, 10, N, 12, 13, 14, N]),
        ("INT64", longs),
        ("FLOAT32", [10.1, 20, -1, 3.1415, -60, N, 1, 2, 3, 4, 5, N, 7, 8, 9, 10, 11, N, 13, 14, 15]),
        ("FLOAT32", [10.1, 20, -2, 3.1415, -60, -50, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15]),
        ("FLOAT64", [10.1, 20.0, 33.1, 3.1415, -60.5, N, 1, 2, 3, 4, 5, 6, N, 8, 9, 10, 11, 12, N, 14, 15]),
        ("FLOAT32", [N] * 21),
        ("TS_DAYS", [99, 100, 101, 102, 103, 104, 1, 2, 3, 4, 5, 6, 7, N, 9, 10, 11, 12, 13, N, 15]),
        ("TS_MS", [9, 1006, 101, 5092, N, 88, 1, 2, 3, 4, 5, 6, 7, 8, N, 10, 11, 12, 13, 14, 15]),
        ("TS_S", [1, N, 3, 4, 5, 6, 1, 2, 3, 4, 5, 6, 7, 8, 9, N, 11, 12, 13, 14, 15]),
        (("DEC32", -3), odd_nulls),
        (("DEC64", -8), longs),
        (("DEC128", -2), longs),
        ("STRING", ["A", "B", "C", "D", N, "TESTING", "1", "2", "3", "4", "5", "6", "7", N, "9", "10", "11", "12", "13", N, "15"]),
        ("STRING", ["A", "A", "C", "C", "E", "TESTING", "1", "2", "3", "4", "5", "6", "7", "", "9", "10", "11", "12", "13", "", "15"]),
        ("STRING", [""] * 21),
        ("STRING", ["", N, "", "", N] + [""] * 16),
        ("STRING", [N] * 21),
        (map_struct, [_kv(("1", "2")), _kv(("3", "4")), N, N, _kv(("key", "value"), ("a", "b")), N, N, _kv(("3", "4"), ("1", "2")), [],
                      _kv(None, ("foo", "bar")), _kv(None, None, None), N, N, N, N, N, N, N, N, N, _kv(("the", "end"))]),
        (struct_t, [(1, 1.0), N, (2, 3.0), N, (8, 7.0), (0, 0.0), N, N, (-1, -1.0), (-100, -100.0), (INT_MAX, FLT_MAX), N, N, N, N, N, N,
                    N, N, N, (INT_MIN, FLT_MIN)]),
        (("LIST", "INT32"), [[1, 2], N, [3, 4, N, 5, N], N, N, [6, 7, 8], [N, N, N], [1, 2, 3], [4, 5, 6], [7, 8, 9], [10, 11, 12], [N],
                             [14, N], [14, 15, N, 16, 17, 18], [19, 20, 21], [22, 23, 24], [25, 26, 27], [28, 29, 30], [31, 32, 33], N,
                             [37, 38, 39]]),
        (("LIST", "INT32"), [[]] * 21),
        (("LIST", "INT32"), null_lists),
        ("INT32", [N] * 21),
        (("LIST", "STRING"), [["1", "2", "3"], ["4"], ["5"], ["6, 7"], ["", "9", N], ["11"], [""], [N, N], ["15", N], N, N,
                              ["18", "19", "20"], N, ["22"], ["23", ""], N, N, N, N, [], ["the end"]]),
        (("LIST", "STRING"), [[]] * 21),
        (("LIST", "STRING"), null_lists),
        ("STRING", [N] * 21),
        (list_map, [[_kv(("k1", "v1"), ("k2", "v2")), _kv(("k3", "v3"))],
                    [_kv(("k4", "v4"), ("k5", "v5"), ("k6", "v6")), _kv(("k7", "v7"))],
                    N, N, N,
                    [_kv(("k8", "v8"), ("k9", "v9")), _kv(("k10", "v10"), ("k11", "v11"), ("k12", "v12"), ("k13", "v13"))],
                    [_kv(("k14", "v14"), ("k15", "v15"))], N, N, N, N,
                    [_kv(("k16", "v16"), ("k17", "v17")), _kv(("k18", "v18"))],
                    [_kv(("k19", "v19"), ("k20", "v20")), _kv(("k21", "v21"))],
                    [_kv(("k22", "v22")), _kv(("k23", "v23"))],
                    [N, N, N],
                    [_kv(("k22", N)), _kv(("k23", N))],
                    N, N, N, N, N]),
        (list_date, [_kv((-210, 293), (-719, 205), (-509, 183), (174, 122), (647, 683)), _kv((311, 992), (-169, 482), (166, 525)),
                     _kv((156, 197), (926, 134), (747, 312), (293, 801)), _kv((647, N), (293, 387)), [], N, [], N,
                     _kv((-210, 293), (-719, 205), (-509, 183), (174, 122), (647, 683)), _kv((311, 992), (-169, 482), (166, 525)),
                     _kv((156, 197), (926, 134), (747, 312), (293, 801)), _kv((647, N), (293, 387)), [], N, [], N,
                     _kv((778, 765)), _kv((7, 87), (8, 96)), _kv((9, 56), (10, 532), (11, 456)), N, []]),
    )


def _merge_list_tables():           # testMergeList (:201-236)
    ll = ("LIST", "INT32")
    t1 = table(("INT64", [-881, 482, 660, 896, -129, -108, -428, 0, 617, 782]),
               (ll, [[665], [-267], [398], [-314], [-370], [181], [665, 544], [222], [-587], [544]]))
    t2 = table(("INT64", [-881, 482, 660, 896, 122, 241, 281, 680, 783, None]),
               (ll, [[-370], [398], [-587, 398], [-314], [307], [-397, -633], [-314, 307], [-633], [-397], [181, -919, -175]]))
    want = table(("INT64", [896, -129, -108, -428, 0, 617, 782, 482, 660, 896, 122, 241, 281, 680, 783, None]),
                 (ll, [[-314], [-370], [181], [665, 544], [222], [-587], [544], [398], [-587, 398], [-314], [307], [-397, -633],
                       [-314, 307], [-633], [-397], [181, -919, -175]]))
    return t1, t2, want


def merge_list_case():
    """-> (list of (table, row offset, rows) written as one partition each, the expected merged table)."""
    t1, t2, want = _merge_list_tables()
    return [(t1, 3, 7), (t2, 1, 9)], want


def merge_complex_struct_list_case():   # testMergeComplexStructList (:238-267)
    N = None
    t = table((("LIST", ("LIST", ("STRUCT", ["STRING", "STRING"]))),
               [[_kv(("k1", "v1"), ("k2", "v2")), _kv(("k3", "v3"))], N, [_kv(("k14", "v14"), ("k15", "v15"))], N, [N, N, N],
                [_kv(("k22", N)), _kv(("k23", N))], N, N, N]))
    return [(t, 0, 3), (t, 3, 3), (t, 6, 3)], t


# ---- KudoGpuSerializerTest.java ---------------------------------------------------------------------------------------
def build_medium_table():           # :416-438
    return table(("STRING", ["1", None, "34", "45", "56", "67"]),
                 (("LIST", "INT32"), [[None], [4], [7], None, [], []]),
                 (("STRUCT", ["INT8", "INT64"]), [(None, 11), (2, None), (3, 33), (4, 44), (5, 55), None]),
                 ("INT32", [None, 2, 3, 4, 5, 6]))


def build_half_empty_struct_table():    # :451-465
    return table((("LIST", ("STRUCT", ["INT32"])), [[(1,), (2,), None], [(4,), (5,), (6,)], [(7,), (8,), (9,)], None, [], []]))


def build_string_list_table():      # :506-513
    return table((("LIST", "STRING"), [["*"], ["*"], ["****"], ["", "*", None]]),
                 (("LIST", "STRING"), [[None] * 4, [], [None] * 3, []]))


# every golden table with the slicings its reference test runs
GOLDEN_TABLES = {
    "simple": (build_simple_table, slice_size_loop),
    "empty_struct": (build_empty_struct_table, slice_size_loop),
    "test_table": (build_test_table, slice_size_loop),
    "medium": (build_medium_table, even_slicings),
    "half_empty_struct": (build_half_empty_struct_table, even_slicings),
    "string_list": (build_string_list_table, even_slicings),
}
