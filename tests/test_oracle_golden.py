"""Pins the CPU oracle against the reference's own known-answer vectors (tests/golden) and against the
reference's vendored FarmHash (its stored outputs, and its build in oracle/_ref when there is one).  CPU only."""
import hashlib
import json
import os
import struct

import numpy as np
import pytest

import oracle
from ytsaurus_b200.rowset import U64, Sentinel, EValueType, make_rowset


def _val(d):
    t, v = d["t"], d["v"]
    if t == "int64":
        return int(v)
    if t == "uint64":
        return U64(int(v))
    if t == "double":
        return float(v)
    if t == "boolean":
        return bool(v)
    return v.encode()


def test_fingerprint_golden(golden):
    for case in golden["farm_fingerprint"]["cases"]:
        rs = make_rowset([[_val(case["v0"]), _val(case["v1"])]])
        fps = oracle.value_fingerprints(rs.values, rs.heap)
        assert int(fps[0]) == int(case["fp0"])
        assert int(fps[1]) == int(case["fp1"])
        assert int(oracle.row_fingerprints(rs.values, rs.heap, 2)[0]) == int(case["fp_range"])


def test_null_and_false_collide():
    # unversioned_value.cpp:51-55: Null -> FarmFingerprint(0), Boolean(false) -> FarmFingerprint(0) == 0.
    rs = make_rowset([[None, False]])
    fps = oracle.value_fingerprints(rs.values, rs.heap)
    assert fps[0] == fps[1] == 0


def _seeded(tag, i, n):
    return hashlib.shake_128(f"{tag} {i}".encode()).digest(n)


def _word(tag, i):
    return int.from_bytes(_seeded(tag, i, 8), "little")


def test_farmhash_restatement_matches_reference_build():
    """The reference's outputs on seeded inputs (tests/golden/farmhash_reference.json), and its build (oracle/_ref)
    where one was made from a YTsaurus source tree."""
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "farmhash_reference.json")) as f:
        g = json.load(f)
    ref = oracle.ref_lib()
    xs = [0, 1, 42, 2**63, 2**64 - 1] + [_word("u64", i) for i in range(200)]
    assert len(g["fingerprint_u64"]) == len(xs)
    for x, want in zip(xs, g["fingerprint_u64"]):
        assert oracle.farm_fingerprint_u64(x) == int(want), x
        assert ref is None or ref.ref_fingerprint_u64(x) == int(want), x
    assert len(g["fingerprint_u128"]) == len(g["hash128to64"]) == 200
    for i in range(200):
        lo, hi = _word("u128 lo", i), _word("u128 hi", i)
        want_fp, want_h = int(g["fingerprint_u128"][i]), int(g["hash128to64"][i])
        assert oracle.farm_fingerprint_u128(lo, hi) == want_fp and oracle.lib().yto_hash128to64(lo, hi) == want_h, i
        assert ref is None or (ref.ref_fingerprint_u128(lo, hi) == want_fp and ref.ref_hash128to64(lo, hi) == want_h), i
    # every length class of farmhashna::Hash64: 0, 1-3, 4-7, 8-16, 17-32, 33-64, >64 (incl. multiples of 64)
    lengths = list(range(0, 200)) + [255, 256, 257, 511, 512, 513, 1000, 4096, 65537]
    assert len(g["fingerprint_bytes"]) == len(lengths)
    for n, want in zip(lengths, g["fingerprint_bytes"]):
        b = _seeded("bytes", n, n)
        assert oracle.farm_fingerprint_bytes(b) == int(want), n
        assert ref is None or ref.ref_fingerprint64(b, n) == int(want), n


def test_ordered_partitioner_golden(golden):
    g = golden["ordered_partitioner"]
    bounds = make_rowset([b["prefix"] for b in g["bounds"]], ncols=1)
    blen = [len(b["prefix"]) for b in g["bounds"]]
    binc = [int(b["inclusive"]) for b in g["bounds"]]
    for p in g["probes"]:
        rows = make_rowset([p["row"]])
        idx, _ = oracle.partition_ordered(rows.values, rows.heap, 1, None, bounds.values, bounds.heap, blen, binc)
        assert int(idx[0]) == p["index"], p


def test_hash_partitioner_golden(golden):
    for case in golden["hash_partitioner"]["cases"]:
        for p in case["probes"]:
            rows = make_rowset([p["row"]])
            idx, _ = oracle.partition_hash(rows.values, rows.heap, case["partition_count"],
                                           case["key_column_count"], case["salt"])
            assert int(idx[0]) == p["index"], (case, p)


def test_column_partitioner_errors():
    # partitioner_ut.cpp:69-124 — value of a column is the index; four error classes.
    rows = make_rowset([[U64(3), 5], [U64(0), 6]])
    rows.values["id"][:, 0] = 7
    code, idx = oracle.partition_column(rows.values, 4, 7)
    assert code == 0 and list(idx) == [3, 0]
    assert oracle.partition_column(make_rowset([[1.5]]).values, 4, 0)[0] == 10
    assert oracle.partition_column(make_rowset([[-1]]).values, 4, 0)[0] == 11
    assert oracle.partition_column(make_rowset([[U64(4)]]).values, 4, 0)[0] == 12
    assert oracle.partition_column(make_rowset([[U64(1)]]).values, 4, 9)[0] == 13


def test_type_order_and_nan():
    # row_base.h:11-28 type order; compare-inl.h:49-66 NaN handling; row_ut.cpp:73-86.
    ladder = [Sentinel(EValueType.Min), None, -5, 7, U64(0), U64(2**64 - 1), float("-inf"), -0.0, 1.5,
              float("inf"), float("nan"), False, True, b"", b"a", b"a\x00", b"ab", b"b", b"\xff",
              Sentinel(EValueType.Max)]
    rs = make_rowset([[x] for x in ladder])
    for i in range(len(ladder)):
        for j in range(len(ladder)):
            c = oracle.compare_values(rs.values[i, 0], rs.values[j, 0], rs.heap)
            assert c == (i > j) - (i < j), (ladder[i], ladder[j], c)
    z = make_rowset([[0.0], [-0.0], [float("nan")], [struct.unpack("<d", struct.pack("<Q", 0xFFF8000000000001))[0]]])
    assert oracle.compare_values(z.values[0, 0], z.values[1, 0], z.heap) == 0
    assert oracle.compare_values(z.values[2, 0], z.values[3, 0], z.heap) == 0


def test_any_rejected():
    rs = make_rowset([[b"x"], [b"y"]])
    rs.values["type"][:, 0] = EValueType.Any
    with pytest.raises(oracle.OracleError):
        oracle.compare_values(rs.values[0, 0], rs.values[1, 0], rs.heap)
    with pytest.raises(oracle.OracleError):
        oracle.sort_rows(rs.values, rs.heap, 1)


def test_sort_algorithms_agree_on_keys():
    rng = np.random.default_rng(3)
    rows = [[int(rng.integers(-50, 50)), bytes(rng.integers(97, 100, int(rng.integers(0, 4)), dtype=np.uint8)), i]
            for i in range(25000)]
    rs = make_rowset(rows)
    keys = [(r[0], r[1]) for r in rows]
    expect = sorted(keys)
    for algo in (oracle.SORT_STD, oracle.SORT_STABLE, oracle.SORT_PARTITION_READER):
        perm, _ = oracle.sort_rows(rs.values, rs.heap, 2, None, algo)
        assert sorted(perm.tolist()) == list(range(len(rows)))
        assert [keys[i] for i in perm] == expect
    perm, _ = oracle.sort_rows(rs.values, rs.heap, 2, None, oracle.SORT_STABLE)
    assert perm.tolist() == sorted(range(len(rows)), key=lambda i: keys[i])
    # descending first column (comparator.cpp:56-58)
    perm, _ = oracle.sort_rows(rs.values, rs.heap, 2, [1, 0], oracle.SORT_STABLE)
    assert perm.tolist() == sorted(range(len(rows)), key=lambda i: (-keys[i][0], keys[i][1]))


def test_merge_tie_break_by_stream():
    runs = [[[1, 0], [3, 0], [3, 1]], [[1, 10], [2, 10], [3, 10]], [], [[0, 20], [3, 20]]]
    flat = [r for run in runs for r in run]
    rs = make_rowset(flat)
    off = np.cumsum([0] + [len(r) for r in runs])
    perm = oracle.merge_sorted(rs.values, rs.heap, 1, None, off)
    got = [tuple(flat[i]) for i in perm]
    assert got == [(0, 20), (1, 0), (1, 10), (2, 10), (3, 0), (3, 1), (3, 10), (3, 20)]


def test_decode_integer_value_golden(golden):
    for raw, base, zz, want in golden["decode_integer_value"]["cases"]:
        got = oracle.decode_integer_value(raw, base, zz)
        assert np.int64(np.uint64(got)) == want


def test_string_offsets_golden(golden):
    g = golden["string_offsets"]
    n = len(g["encoded"])
    assert oracle.decode_string_offsets(g["encoded"], g["avg_length"], 0, n).tolist() == g["expected"]
    for i in range(n + 1):
        for j in range(i, n + 1):
            got = oracle.decode_string_offsets(g["encoded"], g["avg_length"], i, j).tolist()
            assert got == [g["expected"][k] - g["expected"][i] for k in range(i, j + 1)]


def test_rle_golden(golden):
    g = golden["rle_decode"]
    for s, e, want in g["cases"]:
        got = oracle.decode_integer_vector(s, e, 0, False, g["values"], rle_idx=g["rle_indexes"])
        assert got.tolist() == want
    rle = golden["rle_translate"]["rle_indexes"]
    for i in range(rle[-1] + 10):
        j = oracle.translate_rle_index(rle, i)
        assert rle[j] <= i and (j == len(rle) - 1 or i < rle[j + 1])


def test_rle_dict_null_bytemap_golden(golden):
    g = golden["rle_dict_nulls"]
    valid = np.zeros(g["total"], dtype=bool)
    for a, b in g["valid_ranges"]:
        valid[a:b] = True
    for s, e in g["windows"]:
        nm = oracle.build_null_bytemap(3, s, e, dict_idx=g["dictionary_indexes"], rle_idx=g["rle_indexes"])
        assert ((nm == 0) == valid[s:e]).all()


def test_bit_pack_roundtrip():
    rng = np.random.default_rng(11)
    for width in [0, 1, 3, 7, 8, 13, 20, 31, 32, 33, 47, 63, 64]:
        mx = (1 << width) - 1 if width else 0
        for n in [0, 1, 5, 64, 65, 1000]:
            vals = rng.integers(0, mx + 1 if width < 63 else 2**63, n, dtype=np.uint64) if width else np.zeros(n, np.uint64)
            if width == 64 and n:
                vals[0] = np.uint64(2**64 - 1)
                mx = 2**64 - 1
            packed = oracle.bit_pack(vals, mx if n else 0)
            if n:
                assert int(packed[0]) >> 56 == (int(mx).bit_length())
            assert (oracle.bit_unpack(packed) == vals).all()


def test_groupby_styles():
    keys = np.array([5, 3, 5, 3, 9, 5], dtype=np.uint64)
    vals = np.array([1, 2, 3, 4, 5, -6], dtype=np.int64)
    vnull = np.array([0, 0, 0, 1, 1, 0], dtype=np.uint8)
    knull = np.array([0, 0, 0, 0, 0, 0], dtype=np.uint8)
    ql = oracle.groupby_sum_count(keys, vals, oracle.VAL_INT64, knull, vnull, style=oracle.STYLE_QL)
    assert ql["keys"].tolist() == [5, 3, 9]  # first-seen order
    assert ql["sum"].view(np.int64).tolist() == [-2, 2, 0]
    assert ql["sum_null"].tolist() == [0, 0, 1]  # group 9 saw only a Null -> sum stays Null (udf/sum.c)
    assert ql["count"].tolist() == [3, 2, 1]
    ch = oracle.groupby_sum_count(keys, vals, oracle.VAL_INT64, knull, vnull, style=oracle.STYLE_CH, threads=3)
    assert ch["keys"].tolist() == [3, 5, 9]
    assert ch["sum"].view(np.int64).tolist() == [2, -2, 0]
    assert ch["count"].tolist() == [2, 3, 1]
    # wrapping uint64 sum (AggregateFunctionSum.h:53-59)
    w = oracle.groupby_sum_count(np.zeros(2, np.uint64), np.array([2**64 - 1, 2], dtype=np.uint64), oracle.VAL_UINT64)
    assert w["sum"].tolist() == [1]


def test_decode_string_pointers_and_lengths_reference_vector():
    """columnar_ut.cpp:281-329 (TDecodeStringsTest.PointersAndLengths): offsets {1,2,3,4,5}, avg 10 -> {0,9,21,28,42,47}."""
    st, ln = oracle.decode_string_pointers_and_lengths([1, 2, 3, 4, 5], 10)
    expected = [0, 9, 21, 28, 42, 47]
    assert st.tolist() == expected[:-1]
    assert ln.tolist() == [expected[i + 1] - expected[i] for i in range(5)]


def test_groupby_two_level_equals_single_level():
    """The multi-threaded ClickHouse-style baseline (two-level, Aggregator.cpp:1486) yields the single-thread answer."""
    rng = np.random.default_rng(8)
    n = 200_000
    k = rng.integers(0, 5000, n, dtype=np.uint64)
    v = rng.integers(-2**40, 2**40, n, dtype=np.int64)
    kn = (rng.random(n) < 0.01).astype(np.uint8)
    vn = (rng.random(n) < 0.05).astype(np.uint8)
    a = oracle.groupby_sum_count(k, v, oracle.VAL_INT64, kn, vn, style=oracle.STYLE_CH, threads=1)
    b = oracle.groupby_sum_count(k, v, oracle.VAL_INT64, kn, vn, style=oracle.STYLE_CH_TWO_LEVEL, threads=4)
    for f in ("keys", "key_null", "sum", "sum_null", "count"):
        assert (a[f] == b[f]).all(), f
