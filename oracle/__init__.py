"""ctypes binding of the CPU ORACLE (oracle/yt_oracle.cpp).

TEST INFRASTRUCTURE ONLY.  Importable from tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference leg; the product package
(ytsaurus_b200) never imports this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libytoracle.so")
_REF_PATH = os.path.join(_HERE, "_ref", "libfarmhash_ref.so")

VALUE_DTYPE = np.dtype(
    [("id", "<u2"), ("type", "u1"), ("flags", "u1"), ("length", "<u4"), ("data", "<u8")]
)
FIXED_COL_DTYPE = np.dtype(
    [("offset", "<u4"), ("width", "<u4"), ("type", "u1"), ("descending", "u1"), ("pad", "u1", (2,))]
)

T_MIN, T_BOTTOM, T_NULL, T_INT64, T_UINT64, T_DOUBLE, T_BOOLEAN = 0x00, 0x01, 0x02, 0x03, 0x04, 0x05, 0x06
T_STRING, T_ANY, T_COMPOSITE, T_MAX = 0x10, 0x11, 0x12, 0xEF


def build(force: bool = False) -> None:
    """Compile the oracle (and oracle/_ref when YTSAURUS_SOURCE_DIR names a YTsaurus source tree)."""
    if force or not os.path.exists(_LIB_PATH) or (
        os.path.getmtime(_LIB_PATH) < os.path.getmtime(os.path.join(_HERE, "yt_oracle.cpp"))
    ):
        subprocess.check_call(["make", "-C", _HERE, "libytoracle.so"])
    src = os.environ.get("YTSAURUS_SOURCE_DIR")
    if src and os.path.isdir(src) and (force or not os.path.exists(_REF_PATH)):
        subprocess.check_call(["make", "-C", _HERE, "ref", f"REF={src}"])


_lib = None
_ref = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB_PATH)
        _lib.yto_farm_fingerprint_u64.restype = C.c_uint64
        _lib.yto_farm_fingerprint_u64.argtypes = [C.c_uint64]
        _lib.yto_farm_fingerprint_u128.restype = C.c_uint64
        _lib.yto_farm_fingerprint_u128.argtypes = [C.c_uint64, C.c_uint64]
        _lib.yto_hash128to64.restype = C.c_uint64
        _lib.yto_hash128to64.argtypes = [C.c_uint64, C.c_uint64]
        _lib.yto_farm_fingerprint_bytes.restype = C.c_uint64
        _lib.yto_farm_fingerprint_bytes.argtypes = [C.c_char_p, C.c_size_t]
        _lib.yto_decode_integer_value.restype = C.c_uint64
        _lib.yto_decode_integer_value.argtypes = [C.c_uint64, C.c_uint64, C.c_int]
        _lib.yto_translate_rle_index.restype = C.c_int64
        _lib.yto_count_ones.restype = C.c_int64
        _lib.yto_bit_pack.restype = C.c_size_t
    return _lib


def ref_lib():
    """The reference's own FarmHash (oracle/_ref), or None when it was never built."""
    global _ref
    if _ref is None and os.path.exists(_REF_PATH):
        _ref = C.CDLL(_REF_PATH)
        _ref.ref_fingerprint64.restype = C.c_uint64
        _ref.ref_fingerprint64.argtypes = [C.c_char_p, C.c_size_t]
        _ref.ref_fingerprint_u64.restype = C.c_uint64
        _ref.ref_fingerprint_u64.argtypes = [C.c_uint64]
        _ref.ref_fingerprint_u128.restype = C.c_uint64
        _ref.ref_fingerprint_u128.argtypes = [C.c_uint64, C.c_uint64]
        _ref.ref_hash128to64.restype = C.c_uint64
        _ref.ref_hash128to64.argtypes = [C.c_uint64, C.c_uint64]
    return _ref


class OracleError(RuntimeError):
    def __init__(self, code: int, what: str):
        super().__init__(f"oracle error {code} in {what}")
        self.code = code


def _p(a, typ=C.c_void_p):
    if a is None:
        return None
    return a.ctypes.data_as(typ)


def _chk(code: int, what: str) -> None:
    if code != 0:
        raise OracleError(code, what)


def _heap(heap) -> np.ndarray:
    if heap is None or len(heap) == 0:
        return np.zeros(1, dtype=np.uint8)
    if isinstance(heap, (bytes, bytearray)):
        return np.frombuffer(bytes(heap), dtype=np.uint8)
    return np.ascontiguousarray(heap, dtype=np.uint8)


def farm_fingerprint_u64(x: int) -> int:
    return lib().yto_farm_fingerprint_u64(x & 0xFFFFFFFFFFFFFFFF)


def farm_fingerprint_u128(lo: int, hi: int) -> int:
    return lib().yto_farm_fingerprint_u128(lo, hi)


def farm_fingerprint_bytes(b: bytes) -> int:
    return lib().yto_farm_fingerprint_bytes(b, len(b))


def value_fingerprints(values: np.ndarray, heap) -> np.ndarray:
    v = np.ascontiguousarray(values.reshape(-1), dtype=VALUE_DTYPE)
    h = _heap(heap)
    out = np.zeros(v.shape[0], dtype=np.uint64)
    _chk(lib().yto_value_fingerprints(_p(v), _p(h), C.c_size_t(v.shape[0]), _p(out)), "value_fingerprints")
    return out


def row_fingerprints(values: np.ndarray, heap, k: int) -> np.ndarray:
    n, c = values.shape
    v = np.ascontiguousarray(values, dtype=VALUE_DTYPE)
    h = _heap(heap)
    out = np.zeros(n, dtype=np.uint64)
    _chk(lib().yto_row_fingerprints(_p(v), _p(h), C.c_size_t(n), C.c_uint32(c), C.c_uint32(k), _p(out)),
         "row_fingerprints")
    return out


def compare_values(a: np.ndarray, b: np.ndarray, heap) -> int:
    a = np.ascontiguousarray(a.reshape(1), dtype=VALUE_DTYPE)
    b = np.ascontiguousarray(b.reshape(1), dtype=VALUE_DTYPE)
    h = _heap(heap)
    out = C.c_int(0)
    _chk(lib().yto_compare_values(_p(a), _p(b), _p(h), C.byref(out)), "compare_values")
    return out.value


def _desc(desc, nkey):
    d = np.zeros(nkey, dtype=np.uint8)
    if desc is not None:
        d[:] = np.asarray(desc, dtype=np.uint8)
    return d


SORT_STD, SORT_STABLE, SORT_PARTITION_READER = 0, 1, 2


def sort_rows(values: np.ndarray, heap, nkey: int, desc=None, algo: int = SORT_STABLE):
    """-> (permutation u32[n], seconds)."""
    n, c = values.shape
    v = np.ascontiguousarray(values, dtype=VALUE_DTYPE)
    h = _heap(heap)
    d = _desc(desc, nkey)
    perm = np.zeros(n, dtype=np.uint32)
    sec = C.c_double(0)
    _chk(lib().yto_sort_rows(_p(v), _p(h), C.c_size_t(n), C.c_uint32(c), C.c_uint32(nkey), _p(d),
                             C.c_int(algo), _p(perm), C.byref(sec)), "sort_rows")
    return perm, sec.value


def partition_ordered(values, heap, nkey, desc, bounds, bounds_heap, bound_len, bound_inclusive):
    n, c = values.shape
    v = np.ascontiguousarray(values, dtype=VALUE_DTYPE)
    h = _heap(heap)
    d = _desc(desc, nkey)
    nb, bc = bounds.shape
    b = np.ascontiguousarray(bounds, dtype=VALUE_DTYPE)
    bh = _heap(bounds_heap)
    bl = np.ascontiguousarray(bound_len, dtype=np.uint32)
    bi = np.ascontiguousarray(bound_inclusive, dtype=np.uint8)
    out = np.zeros(n, dtype=np.int32)
    sec = C.c_double(0)
    _chk(lib().yto_partition_ordered(_p(v), _p(h), C.c_size_t(n), C.c_uint32(c), C.c_uint32(nkey), _p(d),
                                     _p(b), _p(bh), C.c_uint32(nb), C.c_uint32(bc), _p(bl), _p(bi),
                                     _p(out), C.byref(sec)), "partition_ordered")
    return out, sec.value


def partition_hash(values, heap, partition_count: int, key_column_count: int, salt: int = 0):
    n, c = values.shape
    v = np.ascontiguousarray(values, dtype=VALUE_DTYPE)
    h = _heap(heap)
    out = np.zeros(n, dtype=np.int32)
    sec = C.c_double(0)
    _chk(lib().yto_partition_hash(_p(v), _p(h), C.c_size_t(n), C.c_uint32(c), C.c_int32(partition_count),
                                  C.c_int32(key_column_count), C.c_uint64(salt), _p(out), C.byref(sec)),
         "partition_hash")
    return out, sec.value


def partition_column(values, partition_count: int, column_id: int):
    n, c = values.shape
    v = np.ascontiguousarray(values, dtype=VALUE_DTYPE)
    out = np.zeros(n, dtype=np.int32)
    code = lib().yto_partition_column(_p(v), C.c_size_t(n), C.c_uint32(c), C.c_int32(partition_count),
                                      C.c_uint16(column_id), _p(out))
    return code, out


def merge_sorted(values, heap, nkey, desc, run_offsets):
    n, c = values.shape
    v = np.ascontiguousarray(values, dtype=VALUE_DTYPE)
    h = _heap(heap)
    d = _desc(desc, nkey)
    ro = np.ascontiguousarray(run_offsets, dtype=np.uint64)
    perm = np.zeros(n, dtype=np.uint32)
    _chk(lib().yto_merge_sorted(_p(v), _p(h), C.c_uint32(c), C.c_uint32(nkey), _p(d), _p(ro),
                                C.c_uint32(len(ro) - 1), _p(perm)), "merge_sorted")
    return perm


def join_sorted(values, heap, nkey, desc, run_offsets, table_indexes):
    """TSortedJoiningReader: run 0 = primary stream, the others foreign; -> indices of the emitted rows in order."""
    n, c = values.shape
    v = np.ascontiguousarray(values, dtype=VALUE_DTYPE)
    h = _heap(heap)
    d = _desc(desc, nkey)
    ro = np.ascontiguousarray(run_offsets, dtype=np.uint64)
    ti = np.ascontiguousarray(table_indexes, dtype=np.int32)
    assert len(ti) == len(ro) - 1
    perm = np.zeros(max(n, 1), dtype=np.uint32)
    count = C.c_uint64(0)
    _chk(lib().yto_join_sorted(_p(v), _p(h), C.c_uint32(c), C.c_uint32(nkey), _p(d), _p(ro), C.c_uint32(len(ro) - 1),
                               _p(ti), _p(perm), C.byref(count)), "join_sorted")
    return perm[:count.value]


def fixed_cols(cols) -> np.ndarray:
    """cols: iterable of (offset, width, type, descending)."""
    a = np.zeros(len(cols), dtype=FIXED_COL_DTYPE)
    for i, (off, width, typ, desc) in enumerate(cols):
        a[i]["offset"], a[i]["width"], a[i]["type"], a[i]["descending"] = off, width, typ, desc
    return a


def sort_fixed_rows(rows: np.ndarray, row_bytes: int, cols, algo: int = SORT_STD, threads: int = 1):
    """rows: uint8[n*row_bytes].  -> (perm u32[n], seconds of the timed sort region)."""
    rows = np.ascontiguousarray(rows.reshape(-1), dtype=np.uint8)
    n = rows.shape[0] // row_bytes
    fc = fixed_cols(cols)
    perm = np.zeros(n, dtype=np.uint32)
    sec = C.c_double(0)
    _chk(lib().yto_sort_fixed_rows(_p(rows), C.c_size_t(n), C.c_uint32(row_bytes), _p(fc),
                                   C.c_uint32(len(cols)), C.c_int(algo), C.c_int(threads), _p(perm),
                                   C.byref(sec)), "sort_fixed_rows")
    return perm, sec.value


def bit_pack(values: np.ndarray, max_value: int) -> np.ndarray:
    vals = np.ascontiguousarray(values, dtype=np.uint64)
    width = int(max_value).bit_length()
    words = 1 + ((width * len(vals) + 63) >> 6)
    dst = np.zeros(words + 1, dtype=np.uint64)
    used = lib().yto_bit_pack(_p(vals), C.c_size_t(len(vals)), C.c_uint64(max_value), _p(dst))
    return dst[:used].copy()


def bit_unpack(packed: np.ndarray) -> np.ndarray:
    packed = np.ascontiguousarray(packed, dtype=np.uint64)
    size = int(packed[0]) & ((1 << 56) - 1)
    padded = np.concatenate([packed, np.zeros(1, dtype=np.uint64)])
    out = np.zeros(size, dtype=np.uint64)
    lib().yto_bit_unpack(_p(padded), _p(out))
    return out


def decode_integer_vector(start, end, base, zigzag, values, dict_idx=None, rle_idx=None, bitmap=None):
    values = np.ascontiguousarray(values, dtype=np.uint64)
    di = None if dict_idx is None else np.ascontiguousarray(dict_idx, dtype=np.uint32)
    ri = None if rle_idx is None else np.ascontiguousarray(rle_idx, dtype=np.uint64)
    bm = None if bitmap is None else np.ascontiguousarray(bitmap, dtype=np.uint8)
    out = np.zeros(end - start, dtype=np.uint64)
    lib().yto_decode_integer_vector(C.c_int64(start), C.c_int64(end), C.c_uint64(base), C.c_int(int(zigzag)),
                                    _p(di), _p(ri), C.c_int64(0 if ri is None else len(ri)), _p(bm),
                                    _p(values), _p(out))
    return out


def build_null_bytemap(mode, start, end, bitmap=None, dict_idx=None, rle_idx=None):
    di = None if dict_idx is None else np.ascontiguousarray(dict_idx, dtype=np.uint32)
    ri = None if rle_idx is None else np.ascontiguousarray(rle_idx, dtype=np.uint64)
    bm = None if bitmap is None else np.ascontiguousarray(bitmap, dtype=np.uint8)
    out = np.zeros(end - start, dtype=np.uint8)
    lib().yto_build_null_bytemap(C.c_int(mode), C.c_int64(start), C.c_int64(end), _p(bm), _p(di), _p(ri),
                                 C.c_int64(0 if ri is None else len(ri)), _p(out))
    return out


def decode_string_offsets(enc, avg_length, start, end):
    enc = np.ascontiguousarray(enc, dtype=np.uint32)
    out = np.zeros(end - start + 1, dtype=np.uint32)
    lib().yto_decode_string_offsets(_p(enc), C.c_uint32(avg_length), C.c_int64(start), C.c_int64(end), _p(out))
    return out


def decode_string_pointers_and_lengths(enc, avg_length):
    """DecodeStringPointersAndLengths restated -> (start offsets u32, lengths i32)."""
    enc = np.ascontiguousarray(enc, dtype=np.uint32)
    st, ln = np.zeros(len(enc), dtype=np.uint32), np.zeros(len(enc), dtype=np.int32)
    lib().yto_decode_string_pointers_and_lengths(_p(enc), C.c_uint32(avg_length), C.c_int64(len(enc)), _p(st), _p(ln))
    return st, ln


def decode_integer_value(value, base, zigzag):
    return lib().yto_decode_integer_value(value, base, int(zigzag))


def translate_rle_index(rle, index):
    rle = np.ascontiguousarray(rle, dtype=np.uint64)
    return lib().yto_translate_rle_index(_p(rle), C.c_int64(len(rle)), C.c_int64(index))


def count_ones(bitmap, start, end):
    bm = np.ascontiguousarray(bitmap, dtype=np.uint8)
    return lib().yto_count_ones(_p(bm), C.c_int64(start), C.c_int64(end))



# ---- the remaining helpers of client/table_client/columnar.cpp (validity bitmaps, null bytemaps, dictionary indexes,
# counts) restated as the sequential run walks the reference performs ----
FLAGS_DICTIONARY_ZERO, FLAGS_BITMAP = 0, 1


def _flag_args(kind, data, rle):
    d = np.ascontiguousarray(data, dtype=np.uint32 if kind == FLAGS_DICTIONARY_ZERO else np.uint8)
    r = None if rle is None else np.ascontiguousarray(rle, dtype=np.uint64)
    return d, r, C.c_int64(0 if r is None else len(r))


def build_bitmap_from_flags(kind, data, rle, start, end, negate):
    d, r, nr = _flag_args(kind, data, rle)
    out = np.zeros((end - start + 7) // 8, dtype=np.uint8)
    lib().yto_build_bitmap_from_flags(C.c_int(kind), _p(d), _p(r), nr, C.c_int64(start), C.c_int64(end), C.c_int(int(negate)), _p(out))
    return out


def build_bytemap_from_flags(kind, data, rle, start, end, negate):
    d, r, nr = _flag_args(kind, data, rle)
    out = np.zeros(end - start, dtype=np.uint8)
    lib().yto_build_bytemap_from_flags(C.c_int(kind), _p(d), _p(r), nr, C.c_int64(start), C.c_int64(end), C.c_int(int(negate)), _p(out))
    return out


def count_flags(kind, data, rle, start, end):
    d, r, nr = _flag_args(kind, data, rle)
    f = lib().yto_count_flags
    f.restype = C.c_int64
    return f(C.c_int(kind), _p(d), _p(r), nr, C.c_int64(start), C.c_int64(end))


def build_dictionary_indexes(dict_idx, rle, start, end):
    d = None if dict_idx is None else np.ascontiguousarray(dict_idx, dtype=np.uint32)
    r = None if rle is None else np.ascontiguousarray(rle, dtype=np.uint64)
    out = np.zeros(end - start, dtype=np.uint32)
    lib().yto_build_dictionary_indexes(_p(d), _p(r), C.c_int64(0 if r is None else len(r)), C.c_int64(start), C.c_int64(end), _p(out))
    return out


def count_total_string_length(dict_idx, rle, lengths, start, end):
    d = np.ascontiguousarray(dict_idx, dtype=np.uint32)
    r = np.ascontiguousarray(rle, dtype=np.uint64)
    ln = np.ascontiguousarray(lengths, dtype=np.int32)
    f = lib().yto_count_total_string_length
    f.restype = C.c_int64
    return f(_p(d), _p(r), C.c_int64(len(r)), _p(ln), C.c_int64(start), C.c_int64(end))


def translate_rle_end_index(rle, index):
    rle = np.ascontiguousarray(rle, dtype=np.uint64)
    f = lib().yto_translate_rle_end_index
    f.restype = C.c_int64
    return f(_p(rle), C.c_int64(len(rle)), C.c_int64(index))



def ch_column_to_values(ch_type, data, offsets=None, null_map=None, time_adjustment=0, row_count=None):
    """TCHToYTConverter::ConvertColumnToUnversionedValues restated for simple types -> (status, values[VALUE_DTYPE])."""
    data = np.ascontiguousarray(data)
    n = len(data) if row_count is None else row_count
    off = None if offsets is None else np.ascontiguousarray(offsets, dtype=np.uint64)
    nm = None if null_map is None else np.ascontiguousarray(null_map, dtype=np.uint8)
    out = np.zeros(n, dtype=VALUE_DTYPE)
    code = lib().yto_ch_column_to_values(C.c_int(ch_type), _p(data), _p(off), _p(nm), C.c_int64(time_adjustment), C.c_int64(n), _p(out))
    return code, out



def string_column_to_ch(offsets, avg_length, chars, dict_idx, rle, start, count, filter_hint=None):
    """ConvertStringLikeYTColumnToCHColumn restated -> (chars uint8[], offsets uint64[count]) of a ClickHouse ColumnString."""
    off = np.ascontiguousarray(offsets, dtype=np.uint32)
    ch = np.ascontiguousarray(chars, dtype=np.uint8)
    d = None if dict_idx is None else np.ascontiguousarray(dict_idx, dtype=np.uint32)
    r = None if rle is None else np.ascontiguousarray(rle, dtype=np.uint64)
    f = None if filter_hint is None else np.ascontiguousarray(filter_hint, dtype=np.uint8)
    fn = lib().yto_string_column_to_ch
    fn.restype = C.c_int64
    args = (_p(off), C.c_uint32(avg_length), _p(ch), _p(d), _p(r), C.c_int64(0 if r is None else len(r)), C.c_int64(start), C.c_int64(count), _p(f))
    total = fn(*args, None, None)
    out_chars, out_offsets = np.zeros(total, dtype=np.uint8), np.zeros(count, dtype=np.uint64)
    assert fn(*args, _p(out_chars), _p(out_offsets)) == total
    return out_chars, out_offsets


VAL_INT64, VAL_UINT64, VAL_DOUBLE = 0, 1, 2
STYLE_QL, STYLE_CH, STYLE_CH_TWO_LEVEL = 0, 1, 2


def groupby_sum_count(keys, vals, val_type, key_null=None, val_null=None, filt=None, style=STYLE_CH, threads=1):
    """-> dict(keys, key_null, sum (u64 bit patterns), sum_null, count, seconds)."""
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    n = len(keys)
    vals = np.ascontiguousarray(vals).view(np.uint64)
    kn = None if key_null is None else np.ascontiguousarray(key_null, dtype=np.uint8)
    vn = None if val_null is None else np.ascontiguousarray(val_null, dtype=np.uint8)
    fl = None if filt is None else np.ascontiguousarray(filt, dtype=np.uint8)
    ok = np.zeros(n + 1, dtype=np.uint64)
    okn = np.zeros(n + 1, dtype=np.uint8)
    osum = np.zeros(n + 1, dtype=np.uint64)
    osn = np.zeros(n + 1, dtype=np.uint8)
    ocnt = np.zeros(n + 1, dtype=np.uint64)
    ng = C.c_size_t(0)
    sec = C.c_double(0)
    _chk(lib().yto_groupby_sum_count(_p(keys), _p(kn), _p(vals), _p(vn), _p(fl), C.c_size_t(n),
                                     C.c_int(val_type), C.c_int(style), C.c_int(threads), _p(ok), _p(okn),
                                     _p(osum), _p(osn), _p(ocnt), C.byref(ng), C.byref(sec)), "groupby")
    g = ng.value
    return dict(keys=ok[:g].copy(), key_null=okn[:g].copy(), sum=osum[:g].copy(), sum_null=osn[:g].copy(),
                count=ocnt[:g].copy(), seconds=sec.value)


MINMAX_YQL, MINMAX_QL = 0, 1


def groupby_min_max(keys, vals, val_type, key_null=None, val_null=None, filt=None, style=MINMAX_YQL):
    """-> dict(keys, key_null, min, max (u64 bit patterns), null), ordered by (key_null, key)."""
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    n = len(keys)
    vals = np.ascontiguousarray(vals).view(np.uint64)
    kn = None if key_null is None else np.ascontiguousarray(key_null, dtype=np.uint8)
    vn = None if val_null is None else np.ascontiguousarray(val_null, dtype=np.uint8)
    fl = None if filt is None else np.ascontiguousarray(filt, dtype=np.uint8)
    ok = np.zeros(n + 1, dtype=np.uint64)
    okn = np.zeros(n + 1, dtype=np.uint8)
    omn = np.zeros(n + 1, dtype=np.uint64)
    omx = np.zeros(n + 1, dtype=np.uint64)
    onl = np.zeros(n + 1, dtype=np.uint8)
    ng = C.c_size_t(0)
    _chk(lib().yto_groupby_min_max(_p(keys), _p(kn), _p(vals), _p(vn), _p(fl), C.c_size_t(n), C.c_int(val_type), C.c_int(style),
                                   _p(ok), _p(okn), _p(omn), _p(omx), _p(onl), C.byref(ng)), "groupby_min_max")
    g = ng.value
    return dict(keys=ok[:g].copy(), key_null=okn[:g].copy(), min=omn[:g].copy(), max=omx[:g].copy(), null=onl[:g].copy())


AGG_SUM, AGG_MIN, AGG_MAX, AGG_COUNT, AGG_AVG, AGG_ARGMIN, AGG_ARGMAX, AGG_FIRST = range(8)


def groupby_multi(keys, key_nulls, vals, val_nulls, val_types, aggregates, filt=None):
    """QL GROUP BY over a key tuple with a list of aggregates [(op, column[, by_column])], first-seen order.
    keys / vals: lists of uint64 arrays (bit patterns); *_nulls: lists of uint8 bytemaps or None; val_types: EValueType codes."""
    n = len(keys[0])
    nk, nv, na = len(keys), len(vals), len(aggregates)
    keys = [np.ascontiguousarray(k, dtype=np.uint64) for k in keys]
    vals = [np.ascontiguousarray(v, dtype=np.uint64) for v in vals]
    key_nulls = [np.zeros(n, np.uint8) if x is None else np.ascontiguousarray(x, dtype=np.uint8) for x in (key_nulls or [None] * nk)]
    val_nulls = [np.zeros(n, np.uint8) if x is None else np.ascontiguousarray(x, dtype=np.uint8) for x in (val_nulls or [None] * nv)]
    f = None if filt is None else np.ascontiguousarray(filt, dtype=np.uint8)

    def ptrs(arrs):
        return (C.c_void_p * max(len(arrs), 1))(*[a.ctypes.data for a in arrs])
    ok = [np.zeros(max(n, 1), np.uint64) for _ in range(nk)]
    okn = [np.zeros(max(n, 1), np.uint8) for _ in range(nk)]
    ov = [np.zeros(max(n, 1), np.uint64) for _ in range(na)]
    ovn = [np.zeros(max(n, 1), np.uint8) for _ in range(na)]
    counts = np.zeros(max(n, 1), np.uint64)
    first = np.zeros(max(n, 1), np.uint64)
    vt = np.asarray(val_types, dtype=np.uint8)
    op = np.asarray([a[0] for a in aggregates], dtype=np.int32)
    col = np.asarray([a[1] for a in aggregates], dtype=np.int32)
    by = np.asarray([a[2] if len(a) > 2 else -1 for a in aggregates], dtype=np.int32)
    g = C.c_size_t(0)
    _chk(lib().yto_groupby_multi(ptrs(keys), ptrs(key_nulls), C.c_uint32(nk), ptrs(vals), ptrs(val_nulls), _p(vt), C.c_uint32(nv),
                                 _p(op), _p(col), _p(by), C.c_uint32(na), _p(f) if f is not None else None, C.c_size_t(n),
                                 ptrs(ok), ptrs(okn), ptrs(ov), ptrs(ovn), _p(counts), _p(first), C.byref(g)), "groupby_multi")
    g = g.value
    return dict(keys=[k[:g] for k in ok], key_null=[k[:g] for k in okn], values=[v[:g] for v in ov],
                value_null=[v[:g] for v in ovn], count=counts[:g], first_row=first[:g])


def varuint_encode(v: int) -> bytes:
    out = np.zeros(16, dtype=np.uint8)
    lib().yto_varuint_encode.restype = C.c_uint64
    n = lib().yto_varuint_encode(C.c_uint64(v & 0xFFFFFFFFFFFFFFFF), _p(out))
    return out[:n].tobytes()


def zigzag_encode64(v: int) -> int:
    lib().yto_zigzag_encode64.restype = C.c_uint64
    return lib().yto_zigzag_encode64(C.c_int64(v))


def block_encode(values: np.ndarray, heap, row_value_counts=None) -> np.ndarray:
    """THorizontalBlockWriter restated: -> block bytes (uint8)."""
    n, c = values.shape
    v = np.ascontiguousarray(values, dtype=VALUE_DTYPE)
    h = _heap(heap)
    rc = None if row_value_counts is None else np.ascontiguousarray(row_value_counts, dtype=np.uint32)
    cap = n * 4 + n * (5 + c * 30) + int(v["length"].sum()) + 64
    out = np.zeros(cap, dtype=np.uint8)
    lib().yto_block_encode.restype = C.c_uint64
    used = lib().yto_block_encode(_p(v), _p(h), C.c_size_t(n), C.c_uint32(c), _p(rc), _p(out), C.c_uint64(cap))
    if used == 0 and n:
        raise OracleError(2, "block_encode capacity")
    return out[:used].copy()


def block_decode(block: np.ndarray, row_count: int, value_count: int):
    """THorizontalBlockReader restated: -> (values [rows, value_count] with string data = offset into block, counts)."""
    b = np.ascontiguousarray(block, dtype=np.uint8)
    out = np.zeros((row_count, value_count), dtype=VALUE_DTYPE)
    counts = np.zeros(row_count, dtype=np.uint32)
    _chk(lib().yto_block_decode(_p(b), C.c_uint64(b.size), C.c_uint32(row_count), C.c_uint32(value_count), _p(out),
                                _p(counts)), "block_decode")
    return out, counts


def build_partition_keys(values: np.ndarray, heap, weights, incomplete, partition_count: int, desc=None):
    """BuildPartitionKeysFromSamples restated -> list of (sample index, inclusive, maniac)."""
    n, c = values.shape
    v = np.ascontiguousarray(values, dtype=VALUE_DTYPE)
    h = _heap(heap)
    d = _desc(desc, c)
    w = np.ascontiguousarray(weights, dtype=np.int64)
    inc = np.ascontiguousarray(incomplete, dtype=np.uint8)
    cap = max(partition_count, 2)
    os_, oi, om = np.zeros(cap, np.uint32), np.zeros(cap, np.uint8), np.zeros(cap, np.uint8)
    k = lib().yto_build_partition_keys(_p(v), _p(h), C.c_uint32(n), C.c_uint32(c), _p(d), _p(w), _p(inc),
                                       C.c_int(partition_count), _p(os_), _p(oi), _p(om))
    return [(int(os_[i]), bool(oi[i]), bool(om[i])) for i in range(k)]


INTEGER_SEGMENT_DTYPE = np.dtype([
    ("type", "<u4"), ("row_count", "<u4"), ("chunk_row_count", "<u8"), ("min_value", "<u8"), ("data_offset", "<u8"),
    ("data_bytes", "<u8"), ("part_bytes", "<u8", (3,)), ("values_size", "<u4"), ("ids_size", "<u4"),
    ("row_indexes_size", "<u4"), ("values_width", "u1"), ("ids_width", "u1"), ("row_indexes_width", "u1"), ("direct", "u1"),
])
assert INTEGER_SEGMENT_DTYPE.itemsize == 80
SEGMENT_DICTIONARY_RLE, SEGMENT_DICTIONARY_DENSE, SEGMENT_DIRECT_RLE, SEGMENT_DIRECT_DENSE = 0, 1, 2, 3


def convert_integer_column(values: np.ndarray, column: int, value_type: int):
    """TIntegerColumnConverter<T>::Convert restated -> (words, null bitmap bytes, base value)."""
    n, c = values.shape
    v = np.ascontiguousarray(values, dtype=VALUE_DTYPE)
    out = np.zeros(n, dtype=np.uint64)
    bitmap = np.zeros(8 * ((n + 63) // 64), dtype=np.uint8)
    base = C.c_uint64(0)
    _chk(lib().yto_convert_integer_column(_p(v), C.c_size_t(n), C.c_uint32(c), C.c_uint32(column), C.c_uint8(value_type),
                                          _p(out), _p(bitmap), C.byref(base)), "convert_integer_column")
    return out, bitmap, base.value


def encode_integer_column(values, nulls=None, signed: bool = False, max_segment_values: int = 128 * 1024,
                          chunk_row_offset: int = 0):
    """TUnversionedIntegerColumnWriter restated -> (data bytes, segment descriptors)."""
    raw = np.ascontiguousarray(values).view(np.uint64)
    n = raw.size
    nl = None if nulls is None else np.ascontiguousarray(nulls, dtype=np.uint8)
    seg_cap = max(1, (n + max_segment_values - 1) // max_segment_values)
    cap = 16 * n + 64 * seg_cap + 64
    out = np.zeros(cap, dtype=np.uint8)
    segs = np.zeros(seg_cap, dtype=INTEGER_SEGMENT_DTYPE)
    nbytes, nseg = C.c_uint64(0), C.c_uint32(0)
    _chk(lib().yto_encode_integer_column(_p(raw), _p(nl) if nl is not None else None, C.c_uint64(n), C.c_int(int(signed)),
                                         C.c_uint32(max_segment_values), C.c_uint64(chunk_row_offset), _p(out),
                                         C.c_uint64(cap), C.byref(nbytes), _p(segs), C.c_uint32(seg_cap), C.byref(nseg)),
         "encode_integer_column")
    return out[:nbytes.value].copy(), segs[:nseg.value].copy()


PLAIN_SEGMENT_DTYPE = np.dtype([("row_count", "<u4"), ("reserved", "<u4"), ("chunk_row_count", "<u8"), ("data_offset", "<u8"),
                                ("data_bytes", "<u8"), ("part_bytes", "<u8", (3,))])


def encode_plain_column(values, nulls=None, boolean: bool = False, max_segment_values: int = 128 * 1024, chunk_row_offset: int = 0):
    """The unversioned double (values = 64-bit patterns) / boolean (values = one byte per row) column writers restated
    -> (data bytes, segment descriptors)."""
    raw = np.ascontiguousarray(values, dtype=np.uint8) if boolean else np.ascontiguousarray(values).view(np.uint64)
    n = raw.size
    nl = None if nulls is None else np.ascontiguousarray(nulls, dtype=np.uint8)
    seg_cap = max(1, (n + max_segment_values - 1) // max_segment_values)
    cap = 9 * n + 32 * seg_cap + 64
    out = np.zeros(cap, dtype=np.uint8)
    segs = np.zeros(seg_cap, dtype=PLAIN_SEGMENT_DTYPE)
    nbytes, nseg = C.c_uint64(0), C.c_uint32(0)
    _chk(lib().yto_encode_plain_column(C.c_int(int(boolean)), _p(raw), _p(nl) if nl is not None else None, C.c_uint64(n),
                                       C.c_uint32(max_segment_values), C.c_uint64(chunk_row_offset), _p(out), C.c_uint64(cap),
                                       C.byref(nbytes), _p(segs), C.c_uint32(seg_cap), C.byref(nseg)), "encode_plain_column")
    return out[:nbytes.value].copy(), segs[:nseg.value].copy()


STRING_SEGMENT_DTYPE = np.dtype([
    ("type", "<u4"), ("row_count", "<u4"), ("chunk_row_count", "<u8"), ("data_offset", "<u8"), ("data_bytes", "<u8"),
    ("part_bytes", "<u8", (4,)), ("expected_length", "<u4"), ("offsets_size", "<u4"), ("ids_size", "<u4"),
    ("row_indexes_size", "<u4"), ("offsets_width", "u1"), ("ids_width", "u1"), ("row_indexes_width", "u1"), ("direct", "u1"),
    ("reserved", "<u4")])
assert STRING_SEGMENT_DTYPE.itemsize == 88
STRING_MAX_BUFFER_BYTES = 32 << 20  # string_column_writer.cpp:25


def flatten_strings(values):
    """list of bytes / None -> (heap u8, starts u64, lengths u32, nulls u8)."""
    starts, lengths, nulls = [], [], []
    heap = bytearray()
    for v in values:
        starts.append(len(heap))
        lengths.append(0 if v is None else len(v))
        nulls.append(1 if v is None else 0)
        if v is not None:
            heap += v
    return (np.frombuffer(bytes(heap) or b"\0", dtype=np.uint8).copy(), np.asarray(starts, dtype=np.uint64),
            np.asarray(lengths, dtype=np.uint32), np.asarray(nulls, dtype=np.uint8))


def encode_string_column(heap, starts, lengths, nulls=None, max_segment_values: int = 128 * 1024,
                         max_buffer_bytes: int = STRING_MAX_BUFFER_BYTES, chunk_row_offset: int = 0):
    """TUnversionedStringColumnWriter restated -> (data bytes, segment descriptors)."""
    heap = np.ascontiguousarray(heap, dtype=np.uint8)
    starts = np.ascontiguousarray(starts, dtype=np.uint64)
    lengths = np.ascontiguousarray(lengths, dtype=np.uint32)
    n = starts.size
    nl = None if nulls is None else np.ascontiguousarray(nulls, dtype=np.uint8)
    total = int(lengths.sum())
    seg_cap = max(1, (n + max_segment_values - 1) // max_segment_values + total // max(max_buffer_bytes, 1) + 1)
    cap = total + 16 * n + 128 * seg_cap + 64
    out = np.zeros(cap, dtype=np.uint8)
    segs = np.zeros(seg_cap, dtype=STRING_SEGMENT_DTYPE)
    nbytes, nseg = C.c_uint64(0), C.c_uint32(0)
    _chk(lib().yto_encode_string_column(_p(heap), _p(starts), _p(lengths), _p(nl) if nl is not None else None, C.c_uint64(n),
                                        C.c_uint32(max_segment_values), C.c_uint64(max_buffer_bytes), C.c_uint64(chunk_row_offset),
                                        _p(out), C.c_uint64(cap), C.byref(nbytes), _p(segs), C.c_uint32(seg_cap), C.byref(nseg)),
         "encode_string_column")
    return out[:nbytes.value].copy(), segs[:nseg.value].copy()


def decode_string_segment(data, seg):
    """Reads one string segment back (test helper; follows the reader's view of the parts: string_column_reader.cpp
    :266-520 and DecodeStringPointersAndLengths): -> list of bytes / None."""
    blob = np.ascontiguousarray(data[int(seg["data_offset"]):int(seg["data_offset"] + seg["data_bytes"])])
    parts, o = [], 0
    for b in seg["part_bytes"]:
        parts.append(blob[o:o + int(b)])
        o += int(b)

    def unpack(part):
        return bit_unpack(np.ascontiguousarray(part).view(np.uint64))

    def offsets_of(part):
        enc = unpack(part).astype(np.uint32)
        if enc.size == 0:
            return np.zeros(0, np.int64), np.zeros(0, np.int64)
        st, ln = decode_string_pointers_and_lengths(enc, int(seg["expected_length"]))
        return st.astype(np.int64), ln.astype(np.int64)

    def bits(part, n):
        return np.unpackbits(np.ascontiguousarray(part), bitorder="little")[:n]
    t, n = int(seg["type"]), int(seg["row_count"])
    if t == 3:
        st, ln = offsets_of(parts[0])
        nl = bits(parts[1], n)
        raw = parts[2].tobytes()
        return [None if nl[i] else raw[st[i]:st[i] + ln[i]] for i in range(n)]
    if t == 1:
        ids = unpack(parts[0])
        st, ln = offsets_of(parts[1])
        raw = parts[2].tobytes()
        return [None if ids[i] == 0 else raw[st[ids[i] - 1]:st[ids[i] - 1] + ln[ids[i] - 1]] for i in range(n)]
    rows = unpack(parts[0]).astype(np.int64)
    run_of = np.searchsorted(rows, np.arange(n), side="right") - 1
    if t == 2:
        st, ln = offsets_of(parts[1])
        nl = bits(parts[2], len(rows))
        raw = parts[3].tobytes()
        return [None if nl[r] else raw[st[r]:st[r] + ln[r]] for r in run_of]
    ids = unpack(parts[1])
    st, ln = offsets_of(parts[2])
    raw = parts[3].tobytes()
    return [None if ids[r] == 0 else raw[st[ids[r] - 1]:st[ids[r] - 1] + ln[ids[r] - 1]] for r in run_of]


class BlockAggState(C.Structure):
    """== ytgpu_block_agg_state."""
    _fields_ = [("sum", C.c_uint64), ("min_value", C.c_uint64), ("max_value", C.c_uint64), ("count", C.c_uint64),
                ("count_all", C.c_uint64), ("sum_valid", C.c_uint8), ("min_valid", C.c_uint8), ("max_valid", C.c_uint8),
                ("value_type", C.c_uint8), ("reserved", C.c_uint32)]


def block_agg_state(value_type: int, nullable: bool = True) -> BlockAggState:
    s = BlockAggState()
    lib().yto_block_agg_state_init(C.byref(s), C.c_uint8(value_type), C.c_uint8(int(nullable)))
    return s


def block_combine_all(state: BlockAggState, values, validity=None, offset: int = 0, length=None, nullable: bool = True,
                      filter=None) -> BlockAggState:
    """One AddMany of the sum/avg/min/max/count/count_all block aggregators, sequential as in the reference."""
    v = np.ascontiguousarray(values).view(np.uint64)
    if length is None:
        length = v.size - offset
    val = None if validity is None else np.ascontiguousarray(validity, dtype=np.uint8)
    f = None if filter is None else np.ascontiguousarray(filter, dtype=np.uint8)
    _chk(lib().yto_block_combine_all(_p(v), _p(val) if val is not None else None, C.c_int64(offset), C.c_int64(length),
                                     C.c_uint8(state.value_type), C.c_uint8(int(nullable)),
                                     _p(f) if f is not None else None, C.byref(state)), "block_combine_all")
    return state


def hardware_threads() -> int:
    return int(lib().yto_hardware_threads())
