"""dictionary_encode for the 10 numeric types: a reference restatement pinned against the reference's literal vectors
(vector_hash_test.go; tests/golden/dictionary_encode.json) and against pyarrow, then the GPU kernels (C entry points and
the host mirror's compute.DictionaryEncode) against it."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from arrow_go_b200 import _native as N
from helpers import ALL_TYPES, NP_OF, TYPE_NAME, Dev, pack_bits, ptr, unpack_bits

GOLDEN = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "dictionary_encode.json")))
gpu = pytest.mark.gpu
WIDTHS = {1: 8, 2: 16, 4: 32, 8: 64}
MASK, ENCODE = 0, 1


def ref_dictionary_encode(vals, valid, null_encoding):
    """doAppendNumeric (kernels/vector_hash.go:359-385) driving dictionaryEncodeAction (:144-241) over a memo table keyed
    by the raw bytes of a value, like the memo tables of unique.  Returns (indices int32, index validity, dictionary
    values, dictionary validity)."""
    n = len(vals)
    keys = vals.view(f"u{vals.itemsize}").tolist()
    memo, entries, null_index = {}, [], None       # entries: the row that created each dictionary entry, None = the null
    indices = np.zeros(n, dtype=np.int32)
    index_valid = np.ones(n, dtype=bool)
    for i in range(n):
        if valid is not None and not valid[i]:
            if null_encoding == MASK:              # ObserveNullNotFound(-1) -> appendIndex(0, false) :227-234
                index_valid[i] = False
                continue
            if null_index is None:                 # memo.GetOrInsertNull :374-379
                null_index = len(entries)
                entries.append(None)
            indices[i] = null_index                # ObserveNull*(idx) -> appendIndex(idx, true)
            continue
        j = memo.get(keys[i])                      # memo.GetOrInsert :365-373
        if j is None:
            j = memo[keys[i]] = len(entries)
            entries.append(i)
        indices[i] = j
    dictionary = np.zeros(len(entries), dtype=vals.dtype)   # GetDictionary: the null entry's value bytes are 0
    dict_valid = np.array([e is not None for e in entries], dtype=bool)
    rows = [e for e in entries if e is not None]
    dictionary[dict_valid] = vals[rows]
    return indices, index_valid, dictionary, dict_valid


def col(lst, dt):
    vals = np.array([0 if v is None else v for v in lst], dtype=dt)
    valid = np.array([v is not None for v in lst], dtype=bool)
    return vals, (None if valid.all() else valid)


def as_list(vals, valid):
    return [v if ok else None for v, ok in zip(vals.tolist(), valid)]


def expected_list(lst, dt):
    return [None if e is None else dt.type(e).item() for e in lst]


# ------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("t", ALL_TYPES, ids=lambda t: TYPE_NAME[t])
def test_reference_restatement_matches_literals(t):
    dt = np.dtype(NP_OF[t])
    for case in GOLDEN["cases"]:
        v, valid = col(case["input"], dt)
        for mode, name in ((MASK, "mask"), (ENCODE, "encode")):
            idx, iv, d, dv = ref_dictionary_encode(v, valid, mode)
            assert as_list(idx, iv) == case[name]["indices"], (case["name"], name)
            assert as_list(d, dv) == expected_list(case[name]["dictionary"], dt), (case["name"], name)
    for case in GOLDEN["chunked"]:
        chunks = [col(c, dt) for c in case["input"]]
        v = np.concatenate([c[0] for c in chunks])
        valid = np.concatenate([c[1] if c[1] is not None else np.ones(c[0].size, dtype=bool) for c in chunks])
        for mode, name in ((MASK, "mask"), (ENCODE, "encode")):
            idx, iv, d, dv = ref_dictionary_encode(v, valid, mode)
            assert as_list(idx, iv) == [x for c in case[name]["indices"] for x in c], (case["name"], name)
            assert as_list(d, dv) == expected_list(case[name]["dictionary"], dt), (case["name"], name)


def test_reference_restatement_matches_pyarrow():
    import pyarrow as pa
    import pyarrow.compute as pc
    rng = np.random.default_rng(11)
    for dt in (np.int8, np.int32, np.int64, np.float64):
        for n in (1, 100, 5000):
            v = rng.integers(-40, 40, n).astype(dt)
            valid = rng.random(n) > 0.2
            for mode, name in ((MASK, "mask"), (ENCODE, "encode")):
                idx, iv, d, dv = ref_dictionary_encode(v, valid, mode)
                want = pc.dictionary_encode(pa.array(v, mask=~valid), null_encoding=name)
                assert as_list(idx, iv) == want.indices.to_pylist(), (np.dtype(dt).name, n, name)
                assert as_list(d, dv) == want.dictionary.to_pylist(), (np.dtype(dt).name, n, name)
            # chunked: one dictionary over all chunks, indices across chunk boundaries
            cuts = sorted(rng.integers(0, n, 2).tolist())
            parts = [(v[a:b], valid[a:b]) for a, b in zip([0] + cuts, cuts + [n])]
            want = pc.dictionary_encode(pa.chunked_array([pa.array(p, mask=~m, type=pa.from_numpy_dtype(np.dtype(dt))) for p, m in parts]))
            idx, iv, d, dv = ref_dictionary_encode(v, valid, MASK)
            assert as_list(idx, iv) == [x for c in want.chunks for x in c.indices.to_pylist()]
            assert all(c.dictionary.to_pylist() == as_list(d, dv) for c in want.chunks)


def test_registry_has_dictionary_encode():
    from arrow_go_b200 import compute as pc
    assert "dictionary_encode" in pc.function_names()


@pytest.mark.skipif(os.path.exists("/dev/nvidiactl"), reason="a GPU is present")
def test_entry_points_fail_without_gpu():
    """ensure_init runs first: without a device both flavours return AG_ERR_CUDA and leave every output untouched."""
    v = np.arange(16, dtype=np.int64)
    idx = np.full(16, -7, dtype=np.int32)
    d = np.full(16, -7, dtype=np.int64)
    ln, nn = C.c_int64(-7), C.c_int64(-7)
    st, _ = N.call_status("ag_dictionary_encode", 64, ptr(v), None, 0, 16, MASK, ptr(idx), None, ptr(d), None, C.byref(ln), C.byref(nn))
    assert st == N.AG_ERR_CUDA and (idx == -7).all() and (d == -7).all() and ln.value == -7 and nn.value == -7
    st, _ = N.call_status("ag_dictionary_encode_dev", 64, ptr(v), None, 0, 16, MASK, ptr(idx), None, ptr(d), None, 16, ptr(d), None)
    assert st == N.AG_ERR_CUDA and (idx == -7).all() and (d == -7).all()


# ------------------------------------------------------------------------------------------------- GPU
def gpu_encode(ag, bw, vv, vb, voff, n, mode, dtype):
    idx = np.zeros(max(n, 1), dtype=np.int32)
    iv = np.zeros(n // 8 + 8, dtype=np.uint8)
    d = np.zeros(max(n, 1), dtype=dtype)
    dv = np.zeros(n // 8 + 8, dtype=np.uint8)
    ln, nn = C.c_int64(), C.c_int64()
    ag.call("ag_dictionary_encode", bw, ptr(vv), ptr(vb), voff, n, mode, ptr(idx), ptr(iv), ptr(d), ptr(dv), C.byref(ln), C.byref(nn))
    k = ln.value
    return idx[:n], unpack_bits(iv, 0, n), d[:k], unpack_bits(dv, 0, k), nn.value


def check_against_reference(ag, v, valid, voff, mode, what):
    dt = v.dtype
    bw = WIDTHS[dt.itemsize]
    n = v.size
    vv = np.concatenate([np.zeros(voff, dtype=dt), v])
    vb = pack_bits(valid, voff) if valid is not None else None
    widx, wiv, wd, wdv = ref_dictionary_encode(v, valid, mode)
    gidx, giv, gd, gdv, gnn = gpu_encode(ag, bw, vv, vb, voff, n, mode, dt)
    assert gd.size == wd.size, what
    assert gidx.tobytes() == widx.tobytes(), what
    assert gd.tobytes() == wd.tobytes(), what
    if valid is not None:
        if mode == MASK:
            assert np.array_equal(giv, wiv) and gnn == int((~wiv).sum()), what
        else:
            assert np.array_equal(gdv, wdv) and gnn == 0, what
    else:
        assert gnn == 0, what


@gpu
@pytest.mark.parametrize("t", ALL_TYPES, ids=lambda t: TYPE_NAME[t])
def test_gpu_matches_reference(ag, t):
    dt = np.dtype(NP_OF[t])
    rng = np.random.default_rng(70 + t)
    for n in (1, 31, 33, 1000, 70_001):
        for card in (5, 3000):
            for p_null in (0.0, 0.25):
                hi = min(card, np.iinfo(dt).max) if dt.kind != "f" else card
                v = rng.integers(0, hi, n).astype(dt)
                valid = (rng.random(n) >= p_null) if p_null else None
                voff = int(rng.integers(1, 9))
                for mode in (MASK, ENCODE):
                    check_against_reference(ag, v, valid, voff, mode, (TYPE_NAME[t], n, card, p_null, mode))


@gpu
def test_gpu_edge_keys(ag):
    """Raw-byte equality on floats (-0.0 != +0.0, a NaN matches the same NaN), the all-ones key that cannot live in the
    table (uint64 max, int64 -1), and all-null columns under both encodings."""
    rng = np.random.default_rng(5)
    for dt in (np.float32, np.float64):
        v = rng.choice(np.array([np.nan, -0.0, 0.0, np.inf, -np.inf, 1.5], dtype=dt), 5000)
        valid = rng.random(5000) > 0.1
        for mode in (MASK, ENCODE):
            check_against_reference(ag, v, None, 3, mode, (np.dtype(dt).name, mode))
            check_against_reference(ag, v, valid, 3, mode, (np.dtype(dt).name, "nulls", mode))
        idx, _, d, _, _ = gpu_encode(ag, WIDTHS[np.dtype(dt).itemsize], v, None, 0, v.size, MASK, dt)
        assert d.size == 6 and np.signbit(d[(d == 0)]).sum() == 1
    for v in (np.array([7, np.iinfo(np.uint64).max, 7, 3, np.iinfo(np.uint64).max], dtype=np.uint64),
              np.array([-1, 5, -1, 0, 5, -1], dtype=np.int64)):
        for mode in (MASK, ENCODE):
            check_against_reference(ag, v, None, 0, mode, (v.dtype.name, mode))
            check_against_reference(ag, v, np.array([True, False] * (v.size // 2) + [True] * (v.size % 2)), 2, mode, (v.dtype.name, mode))
    for dt in (np.int64, np.uint8, np.float32):
        n = 100
        v = np.zeros(n, dtype=dt)
        valid = np.zeros(n, dtype=bool)
        idx, iv, d, dv, nn = gpu_encode(ag, WIDTHS[np.dtype(dt).itemsize], v, pack_bits(valid), 0, n, MASK, dt)
        assert d.size == 0 and not iv.any() and nn == n and not idx.any()
        idx, iv, d, dv, nn = gpu_encode(ag, WIDTHS[np.dtype(dt).itemsize], v, pack_bits(valid), 0, n, ENCODE, dt)
        assert d.size == 1 and not dv[0] and d.tobytes() == bytes(np.dtype(dt).itemsize) and nn == 0 and not idx.any()


@gpu
def test_gpu_small_table_then_overflow(ag):
    """The two-table scheme of unique, forced down to a 1024-slot first table: columns below and above its capacity give
    the reference's answer; then the shipped policy at 6M rows with 10 and with 3M distinct values."""
    rng = np.random.default_rng(123)
    ag.call("ag_unique_set_policy", 1000, 1024)
    try:
        for dt in (np.int64, np.uint32, np.float64, np.uint8):
            dt = np.dtype(dt)
            for n in (1001, 70_001):
                for card in (5, 400, 520, 3000):
                    for p_null in (0.0, 0.2):
                        hi = min(card, 255) if dt.itemsize == 1 else card
                        v = rng.integers(0, hi, n).astype(dt)
                        if dt.kind == "u":
                            v[rng.integers(0, n, 3)] = np.iinfo(dt).max
                        valid = (rng.random(n) >= p_null) if p_null else None
                        for mode in (MASK, ENCODE):
                            check_against_reference(ag, v, valid, 3, mode, (dt.name, n, card, p_null, mode))
    finally:
        ag.call("ag_unique_set_policy", 0, 0)
    n = 6_000_000
    for card in (10, 3_000_000):
        v = rng.integers(-card // 2, card // 2, n).astype(np.int64)
        dv, idx, d, cnt = Dev(v), Dev(nbytes=n * 4), Dev(nbytes=n * 8), Dev(np.zeros(2, dtype=np.int64))
        ag.call("ag_dictionary_encode_dev", 64, dv.ptr, None, 0, n, MASK, idx.ptr, None, d.ptr, None, n, cnt.ptr, None)
        ag.call("ag_stream_sync", None)
        uniq, first, inverse = np.unique(v, return_index=True, return_inverse=True)
        order = np.argsort(first)
        rank = np.empty_like(order)
        rank[order] = np.arange(order.size)
        k, nulls = (int(x) for x in cnt.get())
        assert k == uniq.size and nulls == 0, card
        assert np.array_equal(d.buf.to_numpy(np.int64, k), v[np.sort(first)]), card
        assert np.array_equal(idx.buf.to_numpy(np.int32, n), rank[inverse].astype(np.int32)), card


@gpu
def test_gpu_100m_rows_on_device(ag):
    """100M int64 rows over 100 values, all on the device: the dictionary is the values in order of first appearance and
    equals unique(); the indices are the inverse map (checked on the host); take(dictionary, indices) gives the column
    back; two calls give byte-identical outputs."""
    n = 100_000_000
    v = Dev(nbytes=n * 8)
    ag.call("ag_generate_dev", 1, 0x17, 0, 99, v.ptr, n, None)
    outs = []
    for _ in range(2):
        idx, d, cnt = Dev(nbytes=n * 4), Dev(nbytes=n * 8), Dev(np.zeros(2, dtype=np.int64))
        ag.call("ag_dictionary_encode_dev", 64, v.ptr, None, 0, n, MASK, idx.ptr, None, d.ptr, None, n, cnt.ptr, None)
        ag.call("ag_stream_sync", None)
        outs.append((idx, d, cnt))
    idx, d, cnt = outs[0]
    k, nulls = (int(x) for x in cnt.get())
    assert k == 100 and nulls == 0
    hv = v.buf.to_numpy(np.int64, n)
    dict_h = d.buf.to_numpy(np.int64, k)
    _, first = np.unique(hv, return_index=True)
    assert np.array_equal(dict_h, hv[np.sort(first)])
    idx_h = idx.buf.to_numpy(np.int32, n)
    assert np.array_equal(dict_h[idx_h], hv)
    uq, ln = Dev(nbytes=n * 8), Dev(np.zeros(2, dtype=np.int64))
    ag.call("ag_unique_dev", 64, v.ptr, None, 0, n, uq.ptr, None, n, ln.ptr, None)
    back = Dev(nbytes=n * 8)
    ag.call("ag_take_primitive_dev", 64, d.ptr, None, 0, k, 32, 1, idx.ptr, None, 0, n, 0, back.ptr, None, None, None)
    ag.call("ag_stream_sync", None)
    assert int(ln.get()[0]) == k and np.array_equal(uq.buf.to_numpy(np.int64, k), dict_h)
    assert np.array_equal(back.buf.to_numpy(np.int64, n), hv)
    idx2, d2, cnt2 = outs[1]
    assert np.array_equal(cnt2.get(), cnt.get())
    assert idx2.buf.to_numpy(np.uint8, n * 4).tobytes() == idx.buf.to_numpy(np.uint8, n * 4).tobytes()
    assert d2.buf.to_numpy(np.uint8, k * 8).tobytes() == d.buf.to_numpy(np.uint8, k * 8).tobytes()


@gpu
def test_gpu_c_entry_points_validate_arguments(ag):
    v = np.arange(64, dtype=np.int64)
    vb = pack_bits(np.ones(64, dtype=bool))
    idx = np.zeros(64, dtype=np.int32); iv = np.zeros(16, dtype=np.uint8)
    d = np.zeros(64, dtype=np.int64); dv = np.zeros(16, dtype=np.uint8)
    ln, nn = C.c_int64(), C.c_int64()

    def host(bw=64, valid=None, off=0, n=64, mode=MASK, ivp=None, dvp=None):
        return N.call_status("ag_dictionary_encode", bw, ptr(v), valid, off, n, mode, ptr(idx), ivp, ptr(d), dvp, C.byref(ln), C.byref(nn))[0]

    assert host(mode=2) == N.AG_ERR_INVALID and host(mode=-1) == N.AG_ERR_INVALID
    assert host(n=-1) == N.AG_ERR_INVALID and host(off=-1) == N.AG_ERR_INVALID
    assert host(valid=ptr(vb), mode=MASK) == N.AG_ERR_INVALID                   # nulls in mask mode need indices_valid
    assert host(valid=ptr(vb), mode=ENCODE) == N.AG_ERR_INVALID                 # nulls in encode mode need dict_valid
    assert host(valid=ptr(vb), mode=MASK, ivp=ptr(iv)) == N.AG_OK and host(valid=ptr(vb), mode=ENCODE, dvp=ptr(dv)) == N.AG_OK
    assert host(bw=1) == N.AG_ERR_NOT_IMPLEMENTED
    assert host(n=0) == N.AG_OK and ln.value == 0 and nn.value == 0
    dvv, didx, dd, cnt = Dev(v), Dev(nbytes=256), Dev(nbytes=512), Dev(np.full(2, 5, dtype=np.int64))
    dvb, div = Dev(vb), Dev(nbytes=64)

    def dev(n=64, off=0, mode=MASK, valid=None, ivp=None, dvp=None, cap=64):
        return N.call_status("ag_dictionary_encode_dev", 64, dvv.ptr, valid, off, n, mode, didx.ptr, ivp, dd.ptr, dvp, cap, cnt.ptr, None)[0]

    assert dev(mode=7) == N.AG_ERR_INVALID and dev(n=-3) == N.AG_ERR_INVALID and dev(cap=-1) == N.AG_ERR_INVALID
    assert dev(valid=dvb.ptr) == N.AG_ERR_INVALID and dev(valid=dvb.ptr, mode=ENCODE) == N.AG_ERR_INVALID
    assert dev(valid=dvb.ptr, ivp=div.ptr) == N.AG_OK
    assert dev(n=0) == N.AG_OK
    ag.call("ag_stream_sync", None)
    assert (cnt.get() == 0).all()


@gpu
def test_gpu_host_mirror_api(ag):
    from arrow_go_b200 import compute as pc
    # array input, both encodings (TestDictionaryEncode with integers standing in for the strings)
    a = pc.Array.from_pylist([7, 9, 7, None, 9, None], pc.INT64)
    r = pc.DictionaryEncode(a)
    assert r.type == pc.DICTIONARY and r.kind == pc.KIND_ARRAY
    assert r.to_pylist() == [0, 1, 0, None, 1, None] and r.null_count == 2
    assert r.dictionary().type == pc.INT64 and r.dictionary().to_pylist() == [7, 9]
    r = pc.DictionaryEncode(a, pc.NULL_ENCODING_ENCODE)
    assert r.to_pylist() == [0, 1, 0, 2, 1, 2] and r.null_count == 0 and r.dictionary().to_pylist() == [7, 9, None]
    # chunked input: TestDictionaryEncodeChunked, chunk lengths kept, one dictionary
    c = pc.Chunked([pc.Array.from_pylist([1, 2, 1], pc.INT32), pc.Array.from_pylist([2, 3, None], pc.INT32)], pc.INT32)
    r = pc.DictionaryEncode(c)
    assert r.kind == pc.KIND_CHUNKED and r.type == pc.DICTIONARY
    chunks = r.chunks()
    assert [len(ch) for ch in chunks] == [3, 3]
    assert [ch.to_pylist() for ch in chunks] == [[0, 1, 0], [1, 2, None]]
    assert all(ch.dictionary().to_pylist() == [1, 2, 3] for ch in chunks)
    rng = np.random.default_rng(9)
    parts = [rng.integers(0, 50, m).astype(np.uint16) for m in (1000, 0, 37, 4000)]
    c = pc.Chunked([pc.Array.from_numpy(p) for p in parts], pc.UINT16)
    r = pc.DictionaryEncode(c)
    widx, _, wd, _ = ref_dictionary_encode(np.concatenate(parts), None, MASK)
    assert [len(ch) for ch in r.chunks()] == [p.size for p in parts]
    assert np.array_equal(np.concatenate([ch.to_numpy()[0] for ch in r.chunks()]), widx)
    assert all(np.array_equal(ch.dictionary().to_numpy()[0], wd) for ch in r.chunks())
    # a dictionary input comes back as it is
    again = pc.DictionaryEncode(pc.DictionaryEncode(a))
    assert again.type == pc.DICTIONARY and again.to_pylist() == [0, 1, 0, None, 1, None] and again.dictionary().to_pylist() == [7, 9]
    # empty input
    e = pc.DictionaryEncode(pc.Array.from_numpy(np.zeros(0, dtype=np.float32)))
    assert len(e) == 0 and len(e.dictionary()) == 0
    # errors: a bad encoding, a boolean input
    with pytest.raises(pc.ArrowError) as ei:
        pc.DictionaryEncode(a, 99)
    assert ei.value.sentinel == "ErrInvalid"
    with pytest.raises(pc.ArrowError) as ei:
        pc.DictionaryEncode(pc.Array.from_pylist([True, False], pc.BOOL))
    assert ei.value.sentinel == "ErrNotImplemented"
    # no other function reads a dictionary array as its int32 indices
    enc = pc.DictionaryEncode(pc.Array.from_pylist([5, 6, 5], pc.INT32))
    i32 = pc.Array.from_pylist([1, 2, 3], pc.INT32)
    mask = pc.Array.from_pylist([True, False, True], pc.BOOL)
    idx = pc.Array.from_pylist([0, 1], pc.INT32)
    calls = [lambda: pc.Add(enc, i32), lambda: pc.Add(i32, enc), lambda: pc.Filter(enc, mask), lambda: pc.Take(enc, idx),
             lambda: pc.Take(i32, enc), lambda: pc.Unique(enc), lambda: pc.SortIndices(enc), lambda: pc.Cast(enc, pc.INT64),
             lambda: pc.Cast(enc, pc.DICTIONARY), lambda: pc.CallFunction("greater", [enc, i32]),
             lambda: pc.CumulativeSum(enc), lambda: pc.export_device(enc),
             lambda: pc.Take(pc.Chunked([enc, enc], pc.DICTIONARY), idx)]
    for k, call in enumerate(calls):
        with pytest.raises(pc.ArrowError):
            call()
            raise AssertionError(f"call {k} returned a result")
