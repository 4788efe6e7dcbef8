"""Round-2 parity tests (GPU, through the C ABI): sorted-input segmented reduce, first-row indices of GROUP BY (QL
emission order), hint-as-hint table sizing, the in-box shuffle entry points on one rank, context options, contexts on
several devices in one process."""
import numpy as np
import pytest

import oracle
from ytsaurus_b200 import capi
from ytsaurus_b200.rowset import EValueType as T

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from ytsaurus_b200 import GpuContext
    c = GpuContext(0)
    yield c
    c.close()


def _sorted_rows(rng, n, groups, vtype):
    import torch
    keys = np.sort(rng.integers(0, groups, n, dtype=np.uint64))
    if groups > 5:
        keys[keys == 3] = np.uint64(2**64 - 1)  # the largest key forms the last group
        keys = np.sort(keys)
    if vtype == oracle.VAL_DOUBLE:
        vals = rng.random(n)
    elif vtype == oracle.VAL_INT64:
        vals = rng.integers(-2**62, 2**62, n, dtype=np.int64)
    else:
        vals = rng.integers(0, 2**64 - 1, n, dtype=np.uint64)
    rows = rng.integers(0, 2**63, (n, 8), dtype=np.int64)
    rows[:, 0] = keys.view(np.int64)
    rows[:, 1] = vals.view(np.int64)
    return keys, vals, torch.from_numpy(rows).cuda().view(torch.uint8).reshape(-1)


@pytest.mark.parametrize("vtype,yt", [(oracle.VAL_INT64, capi.TYPE_INT64), (oracle.VAL_UINT64, capi.TYPE_UINT64), (oracle.VAL_DOUBLE, capi.TYPE_DOUBLE)])
@pytest.mark.parametrize("n,groups", [(1, 1), (5000, 1), (5000, 5000), (300_000, 7), (300_000, 40_000), (2049, 100)])
def test_reduce_sorted_matches_oracle_groupby(ctx, vtype, yt, n, groups):
    import torch
    rng = np.random.default_rng(n + groups + vtype)
    keys, vals, rows = _sorted_rows(rng, n, groups, vtype)
    cap = n + 1
    ok, os_, oc = (torch.zeros(cap, dtype=torch.int64, device="cuda") for _ in range(3))
    g = ctx.reduce_sorted_fixed_rows(rows, 64, 0, 8, yt, ok, os_, oc)
    want = oracle.groupby_sum_count(keys, vals, vtype, style=oracle.STYLE_CH)
    assert g == len(want["keys"])
    assert ok[:g].cpu().numpy().view(np.uint64).tolist() == want["keys"].tolist()
    assert oc[:g].cpu().numpy().view(np.uint64).tolist() == want["count"].tolist()
    if vtype == oracle.VAL_DOUBLE:
        # SUM(double) is order dependent in the reference itself (SURVEY §8c): tolerance 1e-12 * sum|x|
        assert np.allclose(os_[:g].cpu().numpy().view(np.float64), want["sum"].view(np.float64), rtol=1e-12, atol=1e-9)
    else:
        assert os_[:g].cpu().numpy().view(np.uint64).tolist() == want["sum"].tolist()


def test_reduce_sorted_reports_capacity_and_bad_arguments(ctx):
    import torch
    rng = np.random.default_rng(2)
    keys, vals, rows = _sorted_rows(rng, 10_000, 500, oracle.VAL_INT64)
    small = [torch.zeros(10, dtype=torch.int64, device="cuda") for _ in range(3)]
    with pytest.raises(capi.YtGpuError) as e:
        ctx.reduce_sorted_fixed_rows(rows, 64, 0, 8, capi.TYPE_INT64, *small)
    assert e.value.code == capi.ERR_INVALID_ARGUMENT and "capacity" in e.value.message
    big = [torch.zeros(1000, dtype=torch.int64, device="cuda") for _ in range(3)]
    with pytest.raises(capi.YtGpuError):
        ctx.reduce_sorted_fixed_rows(rows, 64, 4, 8, capi.TYPE_INT64, *big)  # misaligned key offset
    with pytest.raises(capi.YtGpuError) as e:
        ctx.reduce_sorted_fixed_rows(rows, 64, 0, 8, capi.TYPE_STRING, *big)
    assert e.value.code == capi.ERR_UNSUPPORTED
    # the context stays usable
    assert ctx.reduce_sorted_fixed_rows(rows, 64, 0, 8, capi.TYPE_INT64, *big) == len(np.unique(keys))


@pytest.mark.parametrize("groups,hint", [(300, 300), (300, 0), (50_000, 50_000), (50_000, 0)])
def test_groupby_first_rows_give_ql_first_seen_order(ctx, groups, hint):
    """YT QL emits groups in first-seen order (InsertGroupRow, cg_routines/registry.cpp:1571-1655): ordering the result
    by first_row reproduces the oracle's QL-style output exactly, NULL-key group included."""
    from ytsaurus_b200 import Column
    rng = np.random.default_rng(groups)
    n = 200_000
    keys = rng.integers(0, groups, n, dtype=np.uint64)
    key_bm = rng.random(n) < 0.01
    vals = rng.integers(-2**40, 2**40, n, dtype=np.int64)
    kcol = Column(T.Uint64, values=keys, null_bitmap=np.packbits(key_bm, bitorder="little"))
    vcol = Column(T.Int64, values=vals.view(np.uint64))
    got = ctx.scan_filter_groupby(kcol, vcol, None, group_count_hint=hint, want_first_rows=True)
    ql = oracle.groupby_sum_count(keys, vals, oracle.VAL_INT64, key_bm, None, style=oracle.STYLE_QL)
    order = np.argsort(got["first_row"], kind="stable")
    assert np.unique(got["first_row"]).size == got["first_row"].size
    assert got["key_null"][order].tolist() == ql["key_null"].tolist()
    nn = ql["key_null"] == 0
    assert got["keys"][order][nn].tolist() == ql["keys"][nn].tolist()
    assert got["sum"][order].tolist() == ql["sum"].tolist() and got["count"][order].tolist() == ql["count"].tolist()
    # and the first row of every group really is its first occurrence
    first_seen = {}
    for i, (k, kn) in enumerate(zip(keys.tolist(), key_bm.tolist())):
        first_seen.setdefault(None if kn else k, i)
    for k, kn, f in zip(got["keys"].tolist(), got["key_null"].tolist(), got["first_row"].tolist()):
        assert first_seen[None if kn else k] == f


@pytest.mark.parametrize("hint", [1, 10, 1500, 3000])
def test_groupby_hint_is_a_hint(ctx, hint):
    """ADVICE r1: a too-small hint must never fail — the shared-memory front table overflows into the global table, a
    full global table is doubled and the pass repeated."""
    from ytsaurus_b200 import Column
    rng = np.random.default_rng(hint)
    n = 400_000
    keys = rng.integers(0, 30_000, n, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)
    vals = rng.integers(-2**62, 2**62, n, dtype=np.int64)
    got = ctx.scan_filter_groupby(Column(T.Uint64, values=keys), Column(T.Int64, values=vals.view(np.uint64)), None,
                                  group_count_hint=hint, capacity=n + 2)
    want = oracle.groupby_sum_count(keys, vals, oracle.VAL_INT64, style=oracle.STYLE_CH)
    assert got["keys"].tolist() == want["keys"].tolist()
    assert got["sum"].tolist() == want["sum"].tolist() and got["count"].tolist() == want["count"].tolist()


def test_shuffle_entry_points_on_one_rank(ctx):
    """ytgpu_shuffle_* with world = 1: sampling, pivot selection, partition/count, scatter and local sort all run (the
    peer of rank 0 is rank 0), so the whole device-side protocol is exercised on the single-GPU box as well."""
    import torch
    import bench
    from ytsaurus_b200.shuffle import NativeShuffleSorter
    rng = np.random.default_rng(9)
    for n in (0, 1, 1000, 150_000):
        rows = rng.integers(0, 2**63, (n, 8), dtype=np.int64)
        rows[:, 0] = rng.integers(0, 5000, n)
        rows[:, 6] = 0
        rows[:, 7] = np.arange(n)
        flat = torch.from_numpy(rows.view(np.uint8).reshape(-1)).cuda()
        s = NativeShuffleSorter(ctx, capacity_rows=n + 16, row_bytes=64)
        for cols, ocols in [([(0, 0, T.Uint64, 0, 1)], [(0, 8, T.Uint64, 0)]),
                            ([(0, 0, T.Uint64, 1, 1), (8, 16, T.String, 0, 1)], [(0, 8, T.Uint64, 1), (8, 16, T.String, 0)])]:
            out, stats = s.sort(flat, 64, cols)
            assert stats.rows_out == n and stats.sent == [n] and stats.received == [n] and out.numel() == n * 64
            if n == 0:
                continue
            want, _ = oracle.sort_fixed_rows(rows.view(np.uint8).reshape(-1, 64), 64, ocols, oracle.SORT_STABLE)
            assert (out.cpu().numpy().reshape(-1, 64) == rows.view(np.uint8).reshape(-1, 64)[want]).all()
            if n:
                assert bench.verify_sort(out, flat, 64, cols)["ok"]
        # capacity errors are reported, not written past the buffer
        if n > 100:
            tiny = NativeShuffleSorter(ctx, capacity_rows=n // 2, row_bytes=64)
            with pytest.raises(capi.YtGpuError) as e:
                tiny.sort(flat, 64, [(0, 0, T.Uint64, 0, 1)])
            assert "capacity" in e.value.message
            tiny.close()
        s.close()


def test_context_option_sort_hybrid(ctx):
    import torch
    from ytsaurus_b200 import GpuContext
    fresh = GpuContext(0)
    assert fresh.get_option("sort_hybrid") == 1  # a new context reports the default it sorts with
    fresh.close()
    rng = np.random.default_rng(3)
    n = 300_000
    rows = rng.integers(0, 2**63, (n, 8), dtype=np.int64)
    flat = torch.from_numpy(rows).cuda().view(torch.uint8).reshape(-1)
    cols = [(0, 0, T.Int64, 0, 1)]
    a, _ = ctx.sort_fixed_rows(flat, 64, cols)
    hybrid_passes = ctx.last_sort_passes()
    ctx.set_option("sort_hybrid", 0)
    b, _ = ctx.sort_fixed_rows(flat, 64, cols)
    full_passes = ctx.last_sort_passes()
    ctx.set_option("sort_hybrid", 1)
    assert bool((a == b).all()) and full_passes == 8 and hybrid_passes < 8
    with pytest.raises(capi.YtGpuError):
        ctx.set_option("no_such_option", 1)


def test_contexts_on_two_devices_in_one_process():
    """ADVICE r1: kernel attributes (dynamic shared memory limits) belong to a device; a job proxy with several GPU slots
    creates contexts on all of them."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    from ytsaurus_b200 import Column, GpuContext
    rng = np.random.default_rng(5)
    n = 200_000
    rows = rng.integers(0, 2**63, (n, 8), dtype=np.int64)
    want, _ = oracle.sort_fixed_rows(rows.view(np.uint8).reshape(-1, 64), 64, [(0, 8, T.Int64, 0)], oracle.SORT_STABLE)
    keys = rng.integers(0, 500, n, dtype=np.uint64)
    vals = rng.integers(-2**40, 2**40, n, dtype=np.int64)
    ref = oracle.groupby_sum_count(keys, vals, oracle.VAL_INT64, style=oracle.STYLE_CH)
    for dev in (1, 0, 1):
        c = GpuContext(dev, use_torch_stream=False)
        flat = torch.from_numpy(rows).to(f"cuda:{dev}").view(torch.uint8).reshape(-1)
        kdev = torch.from_numpy(keys.view(np.int64)).to(f"cuda:{dev}")
        vdev = torch.from_numpy(vals).to(f"cuda:{dev}")
        torch.cuda.synchronize(dev)  # the context runs on its OWN stream: inputs produced on torch's stream must be complete
        out, _ = c.sort_fixed_rows(flat, 64, [(0, 0, T.Int64, 0, 1)])
        assert (out.cpu().numpy().reshape(-1, 64) == rows.view(np.uint8).reshape(-1, 64)[want]).all()
        got = c.scan_filter_groupby(Column(T.Uint64, values=kdev), Column(T.Int64, values=vdev), None, group_count_hint=500)
        assert got["sum"].cpu().tolist() == ref["sum"].view(np.int64).tolist()
        c.close()


def test_decode_string_pointers_and_lengths(ctx):
    """String column reader value decode (string_column_reader.cpp:266-520 -> DecodeStringPointersAndLengths): the
    reference vector of columnar_ut.cpp:281-329 and random segments against the oracle, host and device flavours."""
    import torch
    st, ln = ctx.decode_string_pointers_and_lengths(np.array([1, 2, 3, 4, 5], dtype=np.uint32), 10)
    assert st.tolist() == [0, 9, 21, 28, 42] and ln.tolist() == [9, 12, 7, 14, 5]
    rng = np.random.default_rng(21)
    for n, avg in [(1, 7), (1000, 13), (300_000, 40)]:
        lengths = rng.integers(0, 2 * avg + 1, n)
        ends = np.cumsum(lengths)
        delta = ends - avg * np.arange(1, n + 1)
        enc = ((delta << 1) ^ (delta >> 63)).astype(np.uint32)  # zig-zag
        want_st, want_ln = oracle.decode_string_pointers_and_lengths(enc, avg)
        assert want_ln.tolist() == lengths.tolist()
        st, ln = ctx.decode_string_pointers_and_lengths(enc, avg)
        assert (st == want_st).all() and (ln == want_ln).all()
        st, ln = ctx.decode_string_pointers_and_lengths(torch.from_numpy(enc.view(np.int32)).cuda(), avg)
        assert (st.cpu().numpy().view(np.uint32) == want_st).all() and (ln.cpu().numpy() == want_ln).all()


def test_decode_boolean_and_double_columns(ctx):
    """Boolean segments keep their values in a TBitmap (boolean_column_reader.cpp:134-172), floating-point segments as raw
    64-bit words + null bitmap (floating_point_column_reader.cpp:132-176): both decode through ytgpu_decode_column, with
    dictionary / RLE indexes on top like the integer segments."""
    from ytsaurus_b200 import Column
    rng = np.random.default_rng(4)
    n = 70_001
    bits = rng.random(n) < 0.4
    nulls = rng.random(n) < 0.1
    col = Column(T.Boolean, values=np.packbits(bits, bitorder="little"), bit_width=1, value_count=n,
                 null_bitmap=np.packbits(nulls, bitorder="little"))
    vals, nb = ctx.decode_column(col)
    assert nb.astype(bool).tolist() == nulls.tolist()
    assert vals[~nulls].tolist() == bits[~nulls].astype(np.uint64).tolist() and not vals[nulls].any()
    # RLE over a boolean bitmap
    runs = np.sort(rng.choice(np.arange(1, n), 500, replace=False))
    starts = np.concatenate([[0], runs]).astype(np.uint64)
    rbits = rng.random(len(starts)) < 0.5
    col = Column(T.Boolean, values=np.packbits(rbits, bitorder="little"), bit_width=1, value_count=n, rle_indexes=starts)
    vals, _ = ctx.decode_column(col)
    want = rbits[np.searchsorted(starts, np.arange(n), side="right") - 1]
    assert vals.tolist() == want.astype(np.uint64).tolist()
    # doubles
    d = rng.normal(size=n)
    col = Column(T.Double, values=d.view(np.uint64), null_bitmap=np.packbits(nulls, bitorder="little"))
    vals, nb = ctx.decode_column(col)
    assert (vals.view(np.float64)[~nulls] == d[~nulls]).all() and nb.astype(bool).tolist() == nulls.tolist()


def test_peer_scatter_validates_caller_supplied_indices(ctx):
    """ADVICE r1: ytgpu_scatter_rows_to_peers must not trust partition_index / partition_rows — a value outside
    [0, parts) or counts that disagree with the index would write outside the destination slabs (another GPU's memory)."""
    import torch
    n, parts = 10_000, 4
    rng = np.random.default_rng(1)
    rows = torch.from_numpy(rng.integers(0, 256, n * 64, dtype=np.uint8)).cuda()
    idx = rng.integers(0, parts, n).astype(np.int32)
    counts = np.bincount(idx, minlength=parts)
    dests = [torch.zeros(n * 64, dtype=torch.uint8, device="cuda") for _ in range(parts)]
    ptrs = [d.data_ptr() for d in dests]
    ctx.scatter_rows_to_peers(rows, 64, torch.from_numpy(idx).cuda(), counts.tolist(), ptrs)  # well-formed call works
    got = torch.cat([d[: int(c) * 64] for d, c in zip(dests, counts)]).cpu().numpy().reshape(-1, 64)
    order = np.argsort(idx, kind="stable")
    assert (got == rows.cpu().numpy().reshape(-1, 64)[order]).all()
    # more than 32 partitions take the sort-based path
    idx40 = rng.integers(0, 40, n).astype(np.int32)
    counts40 = np.bincount(idx40, minlength=40)
    dests40 = [torch.zeros(n * 64, dtype=torch.uint8, device="cuda") for _ in range(40)]
    ctx.scatter_rows_to_peers(rows, 64, torch.from_numpy(idx40).cuda(), counts40.tolist(), [d.data_ptr() for d in dests40])
    got = torch.cat([d[: int(c) * 64] for d, c in zip(dests40, counts40)]).cpu().numpy().reshape(-1, 64)
    assert (got == rows.cpu().numpy().reshape(-1, 64)[np.argsort(idx40, kind="stable")]).all()
    bad = idx.copy()
    bad[123] = parts + 3
    with pytest.raises(capi.YtGpuError) as e:
        ctx.scatter_rows_to_peers(rows, 64, torch.from_numpy(bad).cuda(), counts.tolist(), ptrs)
    assert e.value.code == capi.ERR_INVALID_ARGUMENT
    bad[123] = -1
    with pytest.raises(capi.YtGpuError):
        ctx.scatter_rows_to_peers(rows, 64, torch.from_numpy(bad).cuda(), counts.tolist(), ptrs)
    wrong = counts.copy()
    wrong[0] += 5
    wrong[1] -= 5
    with pytest.raises(capi.YtGpuError) as e:
        ctx.scatter_rows_to_peers(rows, 64, torch.from_numpy(idx).cuda(), wrong.tolist(), ptrs)
    assert e.value.code == capi.ERR_INVALID_ARGUMENT


def test_context_notify_fires_after_enqueued_work(ctx):
    """The async boundary (SURVEY §8b "Threading"): a DEVICE-flavour sort is enqueued, then ytgpu_context_notify — the
    callback (what sets the adapter's TFuture) runs only after the sort's output is complete, nobody blocks meanwhile."""
    import ctypes as C
    import threading
    import torch
    n = 2_000_000
    rng = np.random.default_rng(12)
    rows = torch.from_numpy(rng.integers(0, 2**63, (n, 8), dtype=np.int64)).cuda().view(torch.uint8).reshape(-1)
    out = torch.zeros_like(rows)
    fired = threading.Event()
    seen = {}
    CB = C.CFUNCTYPE(None, C.c_void_p)

    def on_done(user):
        seen["user"] = user
        fired.set()

    cb = CB(on_done)
    ctx.sort_fixed_rows(rows, 64, [(0, 0, T.Int64, 0, 1)], want_rows=True, out_rows=out)  # asynchronous: DEVICE buffers
    err = capi.Error()
    capi.check(ctx.lib.ytgpu_context_notify(ctx.handle, C.cast(cb, C.c_void_p), C.c_void_p(42), C.byref(err)), err)
    assert fired.wait(30), "the completion callback never ran"
    assert seen["user"] == 42
    k = out.view(torch.int64).view(-1, 8)[:, 0]  # no synchronize: the callback fired after the gather finished
    assert bool((k[1:] >= k[:-1]).all())


@pytest.mark.parametrize("vkind,yt", [(oracle.VAL_INT64, T.Int64), (oracle.VAL_UINT64, T.Uint64), (oracle.VAL_DOUBLE, T.Double)])
@pytest.mark.parametrize("shape", ["few_groups", "many_groups", "sorted_keys", "rle_keys"])
def test_groupby_min_max(ctx, vkind, yt, shape):
    """MIN / MAX per group beside SUM / COUNT: equal to the row-by-row states of the YQL aggregators (AggLess, NaN the
    biggest: mkql_block_agg_minmax.cpp:20-60) and, on NaN-free data, of QL's min / max UDFs (udf/min.c, max.c); NULL
    values are skipped, a group without values has NULL aggregates; the predicate applies before aggregation."""
    from ytsaurus_b200 import Column
    rng = np.random.default_rng(vkind * 16 + ["few_groups", "many_groups", "sorted_keys", "rle_keys"].index(shape))
    n = 300_000
    groups = {"few_groups": 7, "many_groups": 40_000, "sorted_keys": 900, "rle_keys": 500}[shape]
    keys = rng.integers(0, groups, n, dtype=np.uint64)
    keys[keys == 1] = np.uint64(2**64 - 1)   # the key that equals the table's EMPTY marker
    rle = None
    if shape == "sorted_keys":
        keys = np.sort(keys)
    if shape == "rle_keys":
        keys = np.sort(keys)
        starts = np.flatnonzero(np.r_[True, keys[1:] != keys[:-1]]).astype(np.uint64)
        rle = (keys[starts.astype(np.int64)].copy(), starts)
    key_bm = rng.random(n) < 0.01
    val_bm = rng.random(n) < 0.2
    if shape == "few_groups":
        val_bm[keys == 3] = True   # a group whose values are all NULL
    if vkind == oracle.VAL_DOUBLE:
        vals = rng.standard_normal(n) * 1e6
        vals[rng.random(n) < 0.001] = np.inf
        vals[rng.random(n) < 0.001] = -np.inf
    elif vkind == oracle.VAL_INT64:
        vals = rng.integers(-2**63, 2**63 - 1, n, dtype=np.int64)
    else:
        vals = rng.integers(0, 2**64 - 1, n, dtype=np.uint64)
    if rle is not None:
        kcol = Column(T.Uint64, values=rle[0], rle_indexes=rle[1], value_count=n)
        key_bm[:] = False
    else:
        kcol = Column(T.Uint64, values=keys, null_bitmap=np.packbits(key_bm, bitorder="little"))
    vcol = Column(yt, values=vals.view(np.uint64), null_bitmap=np.packbits(val_bm, bitorder="little"))
    for style, with_nan in ((oracle.MINMAX_YQL, True), (oracle.MINMAX_QL, False)):
        v = vals.copy()
        if with_nan and vkind == oracle.VAL_DOUBLE:
            v[rng.random(n) < 0.01] = np.nan
        vcol = Column(yt, values=v.view(np.uint64), null_bitmap=np.packbits(val_bm, bitorder="little"))
        got = ctx.scan_filter_groupby(kcol, vcol, None, group_count_hint=groups, want_min_max=True)
        want = oracle.groupby_min_max(keys, v, vkind, key_bm, val_bm, style=style)
        sums = oracle.groupby_sum_count(keys, v, vkind, key_bm, val_bm)
        assert got["keys"].tolist() == want["keys"].tolist() and got["key_null"].tolist() == want["key_null"].tolist()
        assert got["sum_null"].tolist() == want["null"].tolist()
        assert got["count"].tolist() == sums["count"].tolist()
        if vkind == oracle.VAL_DOUBLE:
            # NaN comes back as the canonical quiet NaN; everything else bit for bit
            for name in ("min", "max"):
                g, w = got[name].view(np.float64), want[name].view(np.float64)
                assert (np.isnan(g) == np.isnan(w)).all()
                assert (got[name][~np.isnan(w)] == want[name][~np.isnan(w)]).all()
        else:
            assert got["min"].tolist() == want["min"].tolist() and got["max"].tolist() == want["max"].tolist()
            assert got["sum"].tolist() == sums["sum"].tolist()


def test_groupby_min_max_with_predicate_and_device_memory(ctx):
    import torch
    from ytsaurus_b200 import Column
    rng = np.random.default_rng(77)
    n = 1_000_000
    keys = rng.integers(0, 1000, n, dtype=np.uint64)
    vals = rng.integers(-10**9, 10**9, n, dtype=np.int64)
    kcol = Column(T.Uint64, values=torch.from_numpy(keys.view(np.int64)).cuda())
    vcol = Column(T.Int64, values=torch.from_numpy(vals).cuda())
    got = ctx.scan_filter_groupby(kcol, vcol, (capi.CMP_GT, 10**8), group_count_hint=1000, want_min_max=True)
    want = oracle.groupby_min_max(keys, vals, oracle.VAL_INT64, filt=(vals > 10**8).astype(np.uint8))
    assert got["keys"].cpu().numpy().tolist() == want["keys"].tolist()
    assert got["min"].cpu().numpy().tolist() == want["min"].tolist()
    assert got["max"].cpu().numpy().tolist() == want["max"].tolist()
