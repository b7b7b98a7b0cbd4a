"""Known answers of the nested Kudo restatement (tests/kudo_nested_oracle.py) over tables transcribed from the
reference's tests (tests/golden/kudo_nested_golden.py): the 172-byte partition of KudoSerializerTest.testWriteSimple,
split -> assemble = identity for every golden table under every slicing its reference test runs, the two merge known
answers, and agreement with the flat restatement (oracle/kudo.py) on flat tables."""
import struct

import numpy as np
import pytest

import kudo_nested_oracle as K
from golden import kudo_nested_golden as G
from oracle import kudo as KF
from oracle import oracle as O
from util import cols_equal


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


def _write(pieces):
    parts = [K.write_partition(t, off, n) for t, off, n in pieces]
    offs = np.zeros(len(parts) + 1, np.int64)
    np.cumsum([len(p) for p in parts], out=offs[1:])
    return np.frombuffer(b"".join(parts), np.uint8).copy(), offs


def test_write_simple_known_answer():
    """KudoSerializerTest.java:107-133: 4 rows of buildSimpleTable are 172 bytes with these header fields."""
    k = G.SIMPLE_KNOWN
    b = K.write_partition(G.build_simple_table(), 0, 4)
    assert len(b) == k["bytes"]
    magic, off, n, vlen, olen, total, nc = struct.unpack(">7i", b[:28])
    assert (magic, off, n, vlen, olen, total, nc) == (K.MAGIC, k["offset"], k["num_rows"], k["validity_len"], k["offsets_len"],
                                                      k["total_len"], k["num_columns"])
    assert [bool((b[28 + c // 8] >> (c % 8)) & 1) for c in range(nc)] == k["has_validity"]


def test_flatten_simple_table():
    ids, nch, _ = K.flatten(G.build_simple_table())
    assert ids == [O.INT32, O.STRING, O.LIST, O.INT32, O.STRUCT, O.INT8, O.INT64] and nch == [0, 0, 1, 0, 2, 0, 0]


@pytest.mark.parametrize("name", sorted(G.GOLDEN_TABLES))
def test_split_assemble_every_slicing(name):
    build, slicings = G.GOLDEN_TABLES[name]
    t = build()
    ids, nch, scales = K.flatten(t)
    for splits in slicings(t[0].size):
        back = K.assemble_nested(*K.split(t, splits), ids, nch, scales)
        for i, (a, b) in enumerate(zip(t, back)):
            assert tree_equal(a, b), f"{name}: column {i}, splits {splits}"


@pytest.mark.parametrize("case", [G.merge_list_case, G.merge_complex_struct_list_case])
def test_merge_known_answers(case):
    """testMergeList (:201-236), testMergeComplexStructList (:238-267): slices of tables written one partition each and
    merged give the expected table."""
    pieces, want = case()
    ids, nch, scales = K.flatten(want)
    back = K.assemble_nested(*_write(pieces), ids, nch, scales)
    for i, (a, b) in enumerate(zip(want, back)):
        assert tree_equal(a, b), f"column {i}"


def test_flat_tables_match_the_flat_restatement():
    """On a flat table the nested writer gives the bytes of oracle/kudo.py and the nested reader its columns."""
    from util import random_table
    types = [O.INT32, O.STRING, O.DECIMAL128, O.INT8, O.STRING, O.BOOL8]
    cols = random_table(types, 300, seed=11)
    splits = [0, 7, 7, 150, 299, 300]
    buf, offs = K.split(cols, splits)
    want_buf, want_offs = KF.split(cols, splits)
    assert np.array_equal(buf, want_buf) and np.array_equal(offs, want_offs)
    for a, b in zip(KF.assemble(buf, offs, types), K.assemble_nested(buf, offs, types, [0] * len(types))):
        assert tree_equal(a, b)
