"""Python door into the C++ host mirror of arrow-go's compute API (arrow_go_b200/host).

The classes here are thin handles: every call goes through libarrowgpu_host.so
(CallFunction / Add / Filter / Take / Sum restated from the reference) which drives the device
kernels of libarrowgpu.so.  Nothing is computed in Python; numpy is the host container only.

    from arrow_go_b200 import compute as pc
    a = pc.Array.from_pylist([1, None, 3], pc.INT32)
    out = pc.Add(a, pc.Array.from_pylist([4, 5, None], pc.INT32))          # compute.Add (checked)
    out.to_pylist()                                                          # [5, None, None]
    pc.CallFunction("greater", [a, pc.Scalar(2, pc.INT32)])
    pc.Filter(values, mask, null_selection=pc.EMIT_NULLS)
"""
import ctypes as C
import os

import numpy as np

from . import _native as N

_HERE = os.path.dirname(os.path.abspath(__file__))
HOST_LIB_PATH = os.path.join(_HERE, "lib", "libarrowgpu_host.so")

# arrow.Type ids
NA, BOOL, UINT8, INT8, UINT16, INT16, UINT32, INT32, UINT64, INT64, FLOAT16, FLOAT32, FLOAT64 = range(13)
DICTIONARY = 29  # int32 indices + a dictionary (Datum.dictionary()); to_numpy() gives the indices
NP_OF = {UINT8: np.uint8, INT8: np.int8, UINT16: np.uint16, INT16: np.int16, UINT32: np.uint32, INT32: np.int32,
         UINT64: np.uint64, INT64: np.int64, FLOAT32: np.float32, FLOAT64: np.float64}
TYPE_OF_NP = {np.dtype(v): k for k, v in NP_OF.items()}
DROP_NULLS, EMIT_NULLS = 0, 1
KIND_SCALAR, KIND_ARRAY, KIND_CHUNKED = 1, 2, 3


class ArrowError(RuntimeError):
    """Maps ag_status codes onto arrow-go's error sentinels (arrow/errors.go:21-28)."""
    NAMES = {1: "ErrInvalid", 2: "ErrIndex", 3: "ErrNotImplemented", 4: "ErrType", 5: "ErrCUDA", 6: "ErrOOM"}

    def __init__(self, code, msg):
        super().__init__(f"{self.NAMES.get(code, code)}: {msg}")
        self.code = code
        self.sentinel = self.NAMES.get(code, str(code))
        self.msg = msg


_lib = None


def lib():
    global _lib
    if _lib is None:
        N.raw()  # load libarrowgpu.so first (fails loudly if missing)
        if not os.path.exists(HOST_LIB_PATH):
            raise N.NativeError(N.AG_ERR_CUDA, f"{HOST_LIB_PATH} is missing: run __graft_entry__.build()", "load")
        h = C.CDLL(HOST_LIB_PATH)
        p, i, i64 = C.c_void_p, C.c_int, C.c_int64
        pp = C.POINTER(C.c_void_p)
        h.agx_last_error.restype = C.c_char_p
        h.agx_array_from_host.argtypes = [i, i64, i64, p, p, i64, pp]
        h.agx_scalar.argtypes = [i, i, p, pp]
        h.agx_chunked.argtypes = [i, pp, i, pp]
        h.agx_slice.argtypes = [p, i64, i64, pp]
        h.agx_release.argtypes = [p]
        h.agx_release.restype = None
        for nm in ("agx_kind", "agx_type", "agx_has_validity", "agx_num_chunks"):
            getattr(h, nm).argtypes = [p]
        for nm in ("agx_len", "agx_offset", "agx_null_count_raw"):
            getattr(h, nm).argtypes = [p]
            getattr(h, nm).restype = i64
        h.agx_chunk.argtypes = [p, i, pp]
        h.agx_array_to_host.argtypes = [p, p, p, C.POINTER(i64)]
        h.agx_call_function.argtypes = [C.c_char_p, i, i, pp, i, pp]
        h.agx_arith.argtypes = [i, i, p, p, pp]
        h.agx_sum_f64.argtypes = [p, i, C.POINTER(C.c_double)]
        h.agx_sum_i64.argtypes = [p, C.POINTER(i64)]
        h.agx_sum_u64.argtypes = [p, C.POINTER(C.c_uint64)]
        h.agx_iterate_spans.argtypes = [C.POINTER(i64), C.POINTER(i), C.POINTER(i), i, i64, C.POINTER(i64), C.POINTER(i), i, C.POINTER(i)]
        h.agx_function_names.argtypes = [C.c_char_p, i64]
        h.agx_dispatch.argtypes = [C.c_char_p, C.POINTER(i), i]
        h.agx_dispatch_best.argtypes = [C.c_char_p, C.POINTER(i), i]
        h.agx_common_numeric.argtypes = [C.POINTER(i), i]
        h.agx_cast.argtypes = [p, i, i, i, pp]
        h.agx_cumulative_sum.argtypes = [p, i, i, p, pp]
        h.agx_export_device.argtypes = [p, C.POINTER(N.ArrowDeviceArray), C.POINTER(N.ArrowSchema)]
        h.agx_import_device.argtypes = [C.POINTER(N.ArrowDeviceArray), C.POINTER(N.ArrowSchema), pp]
        h.agx_scalar_value.argtypes = [p, C.POINTER(i), p]
        h.agx_sort_indices.argtypes = [p, i, i, pp]
        h.agx_unique.argtypes = [p, pp]
        h.agx_is_in.argtypes = [p, p, i, pp]
        h.agx_dictionary_encode.argtypes = [p, i, pp]
        h.agx_dictionary.argtypes = [p, pp]
        _lib = h
    return _lib


def _check(code):
    if code != 0:
        raise ArrowError(code, lib().agx_last_error().decode("utf-8", "replace"))


class Datum:
    """Owned handle to a host-layer Datum (Array / Chunked / Scalar) whose buffers live in HBM."""

    def __init__(self, handle):
        self._h = handle

    def __del__(self):
        try:
            if self._h:
                lib().agx_release(self._h)
                self._h = None
        except Exception:
            pass

    @property
    def kind(self):
        return lib().agx_kind(self._h)

    @property
    def type(self):
        return lib().agx_type(self._h)

    def __len__(self):
        return int(lib().agx_len(self._h))

    # ---- arrays ----
    @property
    def offset(self):
        return int(lib().agx_offset(self._h))

    @property
    def has_validity(self):
        return bool(lib().agx_has_validity(self._h))

    def slice(self, off, length):
        out = C.c_void_p()
        _check(lib().agx_slice(self._h, off, length, C.byref(out)))
        return Datum(out)

    def chunks(self):
        res = []
        for k in range(lib().agx_num_chunks(self._h)):
            out = C.c_void_p()
            _check(lib().agx_chunk(self._h, k, C.byref(out)))
            res.append(Datum(out))
        return res

    def dictionary(self):
        """The dictionary of a dictionary array (or of one chunk of a dictionary-encoded chunked array)."""
        out = C.c_void_p()
        _check(lib().agx_dictionary(self._h, C.byref(out)))
        return Datum(out)

    def to_numpy(self):
        """(values, valid_bools, null_count) of an Array, or the concatenation over a Chunked.  A dictionary array
        gives its int32 indices."""
        if self.kind == KIND_CHUNKED:
            parts = [c.to_numpy() for c in self.chunks()]
            if not parts:
                dt = np.bool_ if self.type == BOOL else _np_of(self.type)
                return np.zeros(0, dtype=dt), np.zeros(0, dtype=bool), 0
            return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts]), sum(p[2] for p in parts)
        n = len(self)
        vbytes = np.zeros((n + 7) // 8 + 1, dtype=np.uint8)
        nulls = C.c_int64()
        if self.type == BOOL:
            raw = np.zeros((n + 7) // 8 + 1, dtype=np.uint8)
            _check(lib().agx_array_to_host(self._h, raw.ctypes.data, vbytes.ctypes.data, C.byref(nulls)))
            vals = np.unpackbits(raw, bitorder="little")[:n].astype(bool)
        else:
            vals = np.zeros(n, dtype=_np_of(self.type))
            _check(lib().agx_array_to_host(self._h, vals.ctypes.data, vbytes.ctypes.data, C.byref(nulls)))
        valid = np.unpackbits(vbytes, bitorder="little")[:n].astype(bool)
        return vals, valid, int(nulls.value)

    def to_pylist(self):
        vals, valid, _ = self.to_numpy()
        return [(v.item() if ok else None) for v, ok in zip(vals, valid)]

    @property
    def null_count(self):
        return self.to_numpy()[2]


def _np_of(type_id):
    return np.int32 if type_id == DICTIONARY else NP_OF[type_id]


class Array:
    """Constructors for device-resident arrays (array.FromJSON / NewSlice analogues)."""

    @staticmethod
    def from_numpy(values, valid=None, type_id=None, offset=0, null_count=None):
        values = np.ascontiguousarray(values)
        if type_id is None:
            type_id = BOOL if values.dtype == np.bool_ else TYPE_OF_NP[values.dtype]
        n = values.size - offset
        if type_id == BOOL:
            data = np.packbits(values.astype(bool), bitorder="little")
            data = np.concatenate([data, np.zeros(8, dtype=np.uint8)])
        else:
            data = values.astype(NP_OF[type_id], copy=False)
        vptr, vbuf = None, None
        if valid is not None:
            valid = np.asarray(valid, dtype=bool)
            assert valid.size == values.size
            vbuf = np.concatenate([np.packbits(valid, bitorder="little"), np.zeros(8, dtype=np.uint8)])
            vptr = vbuf.ctypes.data
            if null_count is None:
                null_count = int((~valid[offset:]).sum())
        out = C.c_void_p()
        _check(lib().agx_array_from_host(type_id, n, offset, vptr, data.ctypes.data if data.size else None, null_count or 0, C.byref(out)))
        return Datum(out)

    @staticmethod
    def from_pylist(lst, type_id):
        valid = np.array([x is not None for x in lst], dtype=bool)
        dt = np.bool_ if type_id == BOOL else NP_OF[type_id]
        vals = np.array([(False if type_id == BOOL else 0) if x is None else x for x in lst], dtype=dt)
        return Array.from_numpy(vals, None if valid.all() else valid, type_id)


def Scalar(value, type_id):
    """scalar.MakeScalar / MakeNullScalar: value None is a null scalar."""
    out = C.c_void_p()
    if value is None:
        _check(lib().agx_scalar(type_id, 0, None, C.byref(out)))
    else:
        raw = np.array([value], dtype=np.bool_ if type_id == BOOL else NP_OF[type_id])
        _check(lib().agx_scalar(type_id, 1, raw.ctypes.data, C.byref(out)))
    return Datum(out)


def Chunked(chunks, type_id):
    arr = (C.c_void_p * max(len(chunks), 1))(*[c._h for c in chunks])
    out = C.c_void_p()
    _check(lib().agx_chunked(type_id, arr, len(chunks), C.byref(out)))
    d = Datum(out)
    d._keep = chunks
    return d


def CallFunction(name, args, options=None):
    """compute.CallFunction(ctx, name, opts, args...) — options: None, ("arithmetic", no_check_overflow),
    ("filter", null_selection) or ("take", bounds_check)."""
    kind, val = 0, 0
    if options is not None:
        kind = {"arithmetic": 1, "filter": 2, "take": 3}[options[0]]
        val = int(options[1])
    arr = (C.c_void_p * max(len(args), 1))(*[a._h for a in args])
    out = C.c_void_p()
    _check(lib().agx_call_function(name.encode(), kind, val, arr, len(args), C.byref(out)))
    return Datum(out)


def _arith(which, l, r, no_check_overflow):
    out = C.c_void_p()
    _check(lib().agx_arith(which, int(no_check_overflow), l._h, r._h, C.byref(out)))
    return Datum(out)


def Add(l, r, no_check_overflow=False):
    return _arith(0, l, r, no_check_overflow)


def Subtract(l, r, no_check_overflow=False):
    return _arith(1, l, r, no_check_overflow)


def Multiply(l, r, no_check_overflow=False):
    return _arith(2, l, r, no_check_overflow)


def CumulativeSum(values, start=None, skip_nulls=False, checked=False):
    """compute.CumulativeSum / CumulativeSumChecked(ctx, CumulativeOptions{Start, SkipNulls}, values);
    `start` is a Scalar datum (any numeric type: it is safe-cast to the input type) or None."""
    out = C.c_void_p()
    _check(lib().agx_cumulative_sum(values._h, int(checked), int(skip_nulls), start._h if start is not None else None, C.byref(out)))
    return Datum(out)


def export_device(arr):
    """Array datum -> (ArrowDeviceArray, ArrowSchema) sharing the device buffers (zero copy).  The
    consumer (or release_device) must call array.release."""
    da, sc = N.ArrowDeviceArray(), N.ArrowSchema()
    _check(lib().agx_export_device(arr._h, C.byref(da), C.byref(sc)))
    return da, sc


def import_device(device_array, schema):
    """(ArrowDeviceArray, ArrowSchema) -> Array datum; takes ownership of the device array."""
    out = C.c_void_p()
    _check(lib().agx_import_device(C.byref(device_array), C.byref(schema), C.byref(out)))
    return Datum(out)


def Cast(value, to_type, allow_int_overflow=False, allow_float_truncate=False):
    """compute.CastDatum(ctx, value, &CastOptions{ToType, AllowIntOverflow, AllowFloatTruncate}); the
    defaults are SafeCastOptions(to_type) — what implicit promotion uses."""
    out = C.c_void_p()
    _check(lib().agx_cast(value._h, to_type, int(allow_int_overflow), int(allow_float_truncate), C.byref(out)))
    return Datum(out)


def scalar_value(d):
    """(python value or None) of a Scalar datum."""
    valid = C.c_int()
    raw = np.zeros(8, dtype=np.uint8)
    _check(lib().agx_scalar_value(d._h, C.byref(valid), raw.ctypes.data))
    if not valid.value:
        return None
    return raw.view(NP_OF[d.type])[0].item()


def Filter(values, mask, null_selection=DROP_NULLS):
    return CallFunction("filter", [values, mask], ("filter", null_selection))


def Take(values, indices, bounds_check=True):
    return CallFunction("take", [values, indices], ("take", bounds_check))


ASCENDING, DESCENDING = 0, 1
NULLS_AT_END, NULLS_AT_START = 0, 1
NULL_MATCH, NULL_SKIP, NULL_EMIT_NULL, NULL_INCONCLUSIVE = 0, 1, 2, 3


def SortIndices(values, order=ASCENDING, null_placement=NULLS_AT_END):
    """compute.SortIndices(ctx, input, SortOptions): uint64 row indices (arrow/compute/vector_sort.go:205-211)."""
    out = C.c_void_p()
    _check(lib().agx_sort_indices(values._h, int(order), int(null_placement), C.byref(out)))
    return Datum(out)


def Unique(values):
    """compute.Unique: distinct values in order of first appearance (arrow/compute/vector_hash.go)."""
    out = C.c_void_p()
    _check(lib().agx_unique(values._h, C.byref(out)))
    return Datum(out)


def IsIn(values, value_set, null_behavior=NULL_MATCH):
    """compute.IsIn(ctx, SetOptions{ValueSet, NullBehavior}, values) (arrow/compute/scalar_set_lookup.go)."""
    out = C.c_void_p()
    _check(lib().agx_is_in(values._h, value_set._h, int(null_behavior), C.byref(out)))
    return Datum(out)


NULL_ENCODING_MASK, NULL_ENCODING_ENCODE = 0, 1


def DictionaryEncode(values, null_encoding=NULL_ENCODING_MASK):
    """compute.DictionaryEncode(ctx, DictionaryEncodeOptions{NullEncoding}, values) (arrow/compute/vector_hash.go):
    a dictionary array of int32 indices whose dictionary holds the distinct values in order of first appearance.  A
    chunked input gives a chunked output with the same chunk lengths and one shared dictionary."""
    out = C.c_void_p()
    _check(lib().agx_dictionary_encode(values._h, int(null_encoding), C.byref(out)))
    return Datum(out)


class math:
    """arrow/math: Float64.Sum / Int64.Sum / Uint64.Sum (validity ignored, like the reference)."""

    @staticmethod
    def sum_float64(arr, reference_order=False):
        r = C.c_double()
        _check(lib().agx_sum_f64(arr._h, int(reference_order), C.byref(r)))
        return r.value

    @staticmethod
    def sum_int64(arr):
        r = C.c_int64()
        _check(lib().agx_sum_i64(arr._h, C.byref(r)))
        return r.value

    @staticmethod
    def sum_uint64(arr):
        r = C.c_uint64()
        _check(lib().agx_sum_u64(arr._h, C.byref(r)))
        return r.value


def iterate_exec_spans(arg_chunk_lengths, is_chunked, max_chunk_size=(1 << 63) - 1):
    """iterateExecSpans on chunk lengths (metadata only; runs without a GPU).  Returns
    [(pos, len, [chunk index per arg])]."""
    nargs = len(arg_chunk_lengths)
    flat = [x for lens in arg_chunk_lengths for x in lens]
    lens = (C.c_int64 * max(len(flat), 1))(*flat)
    nchunks = (C.c_int * nargs)(*[len(x) for x in arg_chunk_lengths])
    chunked = (C.c_int * nargs)(*[int(b) for b in is_chunked])
    cap = 4096
    out = (C.c_int64 * (2 * cap))()
    idx = (C.c_int * (cap * nargs))()
    n = C.c_int()
    _check(lib().agx_iterate_spans(lens, nchunks, chunked, nargs, max_chunk_size, out, idx, cap, C.byref(n)))
    return [(out[2 * k], out[2 * k + 1], [idx[k * nargs + a] for a in range(nargs)]) for k in range(n.value)]


def function_names():
    buf = C.create_string_buffer(8192)
    _check(lib().agx_function_names(buf, 8192))
    return [x for x in buf.value.decode().split("\n") if x]


def common_numeric(types):
    """commonNumeric (utils.go:178-240): the promoted type id, or None."""
    arr = (C.c_int * len(types))(*types)
    r = lib().agx_common_numeric(arr, len(types))
    return r or None


def dispatch_best(name, types):
    """The input signature `name` would run with after implicit promotion (DispatchBest)."""
    arr = (C.c_int * len(types))(*types)
    _check(lib().agx_dispatch_best(name.encode(), arr, len(types)))
    return list(arr)


def dispatch(name, types):
    arr = (C.c_int * len(types))(*types)
    _check(lib().agx_dispatch(name.encode(), arr, len(types)))
