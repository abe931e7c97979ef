"""ctypes binding of libarrowgpu.so (include/arrowgpu.h).

This module is a plain FFI table: every function is the C-ABI entry point of the same name.
It never falls back to a CPU implementation — if the library is missing or no sm_100 device
is usable the calls fail loudly (NativeError).
"""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libarrowgpu.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "arrowgpu.h")
CDATA_HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "arrowgpu_cdata.h")

# status codes (include/arrowgpu.h)
AG_OK, AG_ERR_INVALID, AG_ERR_INDEX, AG_ERR_NOT_IMPLEMENTED, AG_ERR_TYPE, AG_ERR_CUDA, AG_ERR_OOM = range(7)
NO_ERROR_POS = (1 << 63) - 1

# arrow.Type ids
NULL, BOOL, UINT8, INT8, UINT16, INT16, UINT32, INT32, UINT64, INT64, FLOAT16, FLOAT32, FLOAT64 = range(13)
# ArithmeticOp
OP_ADD, OP_SUB, OP_MUL, OP_DIV, OP_ABS, OP_NEGATE = 0, 1, 2, 3, 4, 5
OP_SIGN, OP_ADD_CHECKED, OP_SUB_CHECKED, OP_MUL_CHECKED, OP_DIV_CHECKED, OP_ABS_CHECKED, OP_NEGATE_CHECKED = 20, 21, 22, 23, 24, 25, 26
OP_BIT_AND, OP_BIT_OR, OP_BIT_XOR, OP_BIT_NOT, OP_SHIFT_LEFT, OP_SHIFT_RIGHT, OP_SHIFT_LEFT_CHECKED, OP_SHIFT_RIGHT_CHECKED = 64, 65, 66, 67, 68, 69, 70, 71
# CompareOperator
CMP_EQ, CMP_NE, CMP_GT, CMP_GE, CMP_LT, CMP_LE = range(6)
SHAPE_AA, SHAPE_AS, SHAPE_SA = range(3)
BITOP_AND, BITOP_OR, BITOP_XOR, BITOP_ANDNOT, BITOP_XNOR = range(5)
KLEENE_AND, KLEENE_OR, KLEENE_ANDNOT = range(3)
DROP_NULLS, EMIT_NULLS = 0, 1


class Span3(C.Structure):
    """ag_span3: one aligned span of a chunked binary call."""
    _fields_ = [("l", C.c_void_p), ("r", C.c_void_p), ("out", C.c_void_p), ("n", C.c_int64)]


def span_table(spans):
    """[(l_ptr, r_ptr, out_ptr, n), ...] -> ctypes array of ag_span3."""
    arr = (Span3 * max(len(spans), 1))()
    for k, (l, r, o, n) in enumerate(spans):
        arr[k].l, arr[k].r, arr[k].out, arr[k].n = l, r, o, n
    return arr


class NativeError(RuntimeError):
    """A C-ABI call returned a non-zero ag_status."""

    def __init__(self, status, message, func):
        super().__init__(f"{func}: status {status}: {message}")
        self.status = status
        self.message = message
        self.func = func


_p = C.c_void_p
_i = C.c_int
_i8 = C.c_int8
_i64 = C.c_int64
_sz = C.c_size_t
_u64 = C.c_uint64
_pi64 = C.POINTER(C.c_int64)

# name -> argtypes.  Every function returns ag_status (int) unless listed in _SPECIAL.
_SIGS = {
    "ag_init": [_i],
    "ag_init_all": [C.POINTER(_i)],
    "ag_set_device": [_i],
    "ag_get_device": [C.POINTER(_i)],
    "ag_shutdown": [],
    "ag_device_count": [C.POINTER(_i)],
    "ag_device_info": [C.POINTER(_i), C.POINTER(_i), C.POINTER(_sz), C.POINTER(_i), C.POINTER(_i)],
    "ag_host_alloc": [C.POINTER(_p), _sz],
    "ag_host_realloc": [C.POINTER(_p), _sz, _sz],
    "ag_host_free": [_p],
    "ag_host_register": [_p, _sz],
    "ag_host_unregister": [_p],
    "ag_dev_alloc": [C.POINTER(_p), _sz],
    "ag_dev_free": [_p],
    "ag_dev_memset": [_p, _i, _sz, _p],
    "ag_upload": [_p, _p, _sz, _p],
    "ag_download": [_p, _p, _sz, _p],
    "ag_copy_dev": [_p, _p, _sz, _p],
    "ag_stream_create": [C.POINTER(_p)],
    "ag_stream_destroy": [_p],
    "ag_stream_sync": [_p],
    "ag_event_create": [C.POINTER(_p)],
    "ag_event_destroy": [_p],
    "ag_event_record": [_p, _p],
    "ag_event_sync": [_p],
    "ag_event_elapsed_ms": [_p, _p, C.POINTER(C.c_float)],
    "ag_flush_l2": [_p],
    # sum
    "ag_sum_f64": [_p, _sz, C.POINTER(C.c_double)],
    "ag_sum_i64": [_p, _sz, C.POINTER(C.c_int64)],
    "ag_sum_u64": [_p, _sz, C.POINTER(C.c_uint64)],
    "ag_sum_f64_reforder": [_p, _sz, C.POINTER(C.c_double)],
    "ag_sum_f64_dev": [_p, _sz, _p, _p],
    "ag_sum_i64_dev": [_p, _sz, _p, _p],
    "ag_sum_u64_dev": [_p, _sz, _p, _p],
    "ag_sum_f64_reforder_dev": [_p, _sz, _p, _p],
    # multi-GPU
    "ag_shard_range": [_i64, _i, _i, _pi64, _pi64],
    "ag_comm_local_handle": [_i, _p],
    "ag_comm_create": [C.POINTER(_p), _i, _i, _p],
    "ag_comm_create_local": [C.POINTER(_p), _i, C.POINTER(_i)],
    "ag_comm_unique_id": [_p],
    "ag_comm_attach_nccl": [_p, _p],
    "ag_comm_info": [_p, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i)],
    "ag_comm_destroy": [_p],
    "ag_sum_i64_global_dev": [_p, _p, _sz, _p, _p],
    "ag_sum_u64_global_dev": [_p, _p, _sz, _p, _p],
    "ag_sum_f64_global_dev": [_p, _p, _sz, _p, _p],
    "ag_sum_i64_global_nccl_dev": [_p, _p, _sz, _p, _p],
    # arithmetic
    "ag_arith_binary": [_i, _i8, _p, _p, _p, _i64],
    "ag_arith_arr_scalar": [_i, _i8, _p, _p, _p, _i64],
    "ag_arith_scalar_arr": [_i, _i8, _p, _p, _p, _i64],
    "ag_arith_unary_same": [_i, _i8, _p, _p, _i64],
    "ag_arith_unary_diff": [_i, _i, _i8, _p, _p, _i64],
    "ag_arith_binary_dev": [_i, _i8, _i, _p, _p, _p, _i64, _p],
    "ag_arith_binary_spans": [_i, _i8, _i, _p, _i64],
    "ag_arith_binary_spans_dev": [_i, _i8, _i, _p, _i64, _p],
    "ag_arith_unary_same_dev": [_i, _i8, _p, _p, _i64, _p],
    "ag_arith_unary_diff_dev": [_i, _i, _i8, _p, _p, _i64, _p],
    "ag_arith_checked": [_i, _i8, _i, _p, _p, _i64, _p, _p, _i64, _p, _i64, _pi64],
    "ag_arith_checked_dev": [_i, _i8, _i, _p, _p, _i64, _p, _p, _i64, _p, _i64, _p, _p],
    "ag_arith_unary_checked": [_i, _i8, _p, _p, _i64, _pi64],
    "ag_arith_unary_checked_dev": [_i, _i8, _p, _p, _i64, _p, _p],
    "ag_error_word_reset_dev": [_p, _p],
    "ag_min_max": [_i, _p, _i64, _p, _p],
    "ag_min_max_dev": [_i, _p, _i64, _p, _p],
    "ag_cumulative_sum": [_i, _p, _p, _i64, _i64, _p, _i, _i, _p, _p, _pi64, _pi64],
    "ag_cumulative_sum_state_init_dev": [_p, _i, _p, _p],
    "ag_cumulative_sum_dev": [_i, _p, _p, _i64, _i64, _i, _i, _p, _p, _i64, _p, _p, _p],
    # numeric casts
    "ag_cast_numeric": [_i, _i, _p, _p, _i64],
    "ag_cast_numeric_dev": [_i, _i, _p, _p, _i64, _p],
    "ag_cast_numeric_checked": [_i, _i, _p, _p, _i64, _p, _i64, _i, _i, _pi64],
    "ag_cast_numeric_checked_dev": [_i, _i, _p, _p, _i64, _p, _i64, _i, _i, _p, _p],
    # compare
    "ag_compare": [_i, _i, _i, _p, _p, _p, _i64, _i],
    "ag_compare_dev": [_i, _i, _i, _p, _p, _p, _i64, _i, _p],
    # bitmaps
    "ag_bitmap_op": [_i, _p, _i64, _p, _i64, _p, _i64, _i64],
    "ag_bitmap_copy": [_p, _i64, _i64, _p, _i64],
    "ag_bitmap_invert": [_p, _i64, _i64, _p, _i64],
    "ag_bitmap_set": [_p, _i64, _i64, _i],
    "ag_bitmap_popcount": [_p, _i64, _i64, _pi64],
    "ag_bitmap_op_dev": [_i, _p, _i64, _p, _i64, _p, _i64, _i64, _p],
    "ag_bitmap_copy_dev": [_p, _i64, _i64, _p, _i64, _p],
    "ag_bitmap_invert_dev": [_p, _i64, _i64, _p, _i64, _p],
    "ag_bitmap_set_dev": [_p, _i64, _i64, _i, _p],
    "ag_bitmap_popcount_dev": [_p, _i64, _i64, _p, _p],
    "ag_kleene": [_i, _p, _p, _i64, _p, _p, _i64, _p, _p, _i64, _i64],
    "ag_kleene_dev": [_i, _p, _p, _i64, _p, _p, _i64, _p, _p, _i64, _i64, _p],
    # filter / take
    "ag_filter_output_size": [_p, _p, _i64, _i64, _i, _pi64],
    "ag_filter_primitive": [_i, _p, _p, _i64, _p, _p, _i64, _i64, _i, _p, _p, _pi64, _pi64],
    "ag_filter_output_size_dev": [_p, _p, _i64, _i64, _i, _p, _p],
    "ag_filter_primitive_dev": [_i, _p, _p, _i64, _p, _p, _i64, _i64, _i, _p, _p, _i64, _p, _p],
    "ag_filter_compare_scalar_dev": [_i, _i, _p, _p, _i64, _p, _i64, _p, _p],
    "ag_take_indices": [_i, _p, _p, _i64, _i64, _i, _p, _p, _pi64],
    "ag_take_indices_dev": [_i, _p, _p, _i64, _i64, _i, _p, _p, _i64, _p, _p],
    "ag_take_primitive": [_i, _p, _p, _i64, _i64, _i, _i, _p, _p, _i64, _i64, _i, _p, _p, _pi64, _pi64, _pi64],
    "ag_take_primitive_dev": [_i, _p, _p, _i64, _i64, _i, _i, _p, _p, _i64, _i64, _i, _p, _p, _p, _p],
    "ag_take_set_policy": [_i, _i64, _i64, _i64],
    "ag_unique_set_policy": [_i64, _i64],
    "ag_is_in": [_i, _p, _p, _i64, _i64, _p, _p, _i64, _i64, _i, _p, _p, _pi64],
    "ag_is_in_dev": [_i, _p, _p, _i64, _i64, _p, _p, _i64, _i64, _i, _p, _p, _p, _p],
    "ag_unique": [_i, _p, _p, _i64, _i64, _p, _p, _pi64, _pi64],
    "ag_unique_dev": [_i, _p, _p, _i64, _i64, _p, _p, _i64, _p, _p],
    "ag_dictionary_encode": [_i, _p, _p, _i64, _i64, _i, _p, _p, _p, _p, _pi64, _pi64],
    "ag_dictionary_encode_dev": [_i, _p, _p, _i64, _i64, _i, _p, _p, _p, _p, _i64, _p, _p],
    "ag_sort_indices": [_i, _p, _p, _i64, _i64, _i, _i, _p, _pi64, _pi64],
    "ag_sort_indices_dev": [_i, _p, _p, _i64, _i64, _i, _i, _p, _pi64, _pi64, _p],
    "ag_parquet_unpack32": [_p, _p, _i64, _i, _pi64],
    "ag_parquet_unpack32_dev": [_p, _p, _i64, _i, _pi64, _p],
    "ag_parquet_bytes_to_bools": [_p, _i64, _p, _i64],
    "ag_parquet_bytes_to_bools_dev": [_p, _i64, _p, _i64, _p],
    "ag_parquet_def_levels_to_bitmap": [_p, _i64, _i, _i, _p, _i64, _i64, _pi64, _pi64],
    "ag_parquet_def_levels_to_bitmap_dev": [_p, _i64, _i, _i, _p, _i64, _i64, _p, _p],
    # parity helpers
    "ag_checksum64_dev": [_p, _sz, _p, _p],
    "ag_generate_dev": [_i, _u64, _i64, _i64, _p, _sz, _p],
}
for _op in ("eq", "ne", "gt", "ge"):
    for _sh in ("aa", "as", "sa"):
        _SIGS[f"ag_cmp_{_op}_{_sh}"] = [_i, _p, _p, _p, _i64, _i]

# Arrow C Data / C Device Data Interface structs (include/arrowgpu_cdata.h)
class ArrowSchema(C.Structure):
    pass


ArrowSchema._fields_ = [("format", C.c_char_p), ("name", C.c_char_p), ("metadata", C.c_char_p), ("flags", C.c_int64),
                        ("n_children", C.c_int64), ("children", C.c_void_p), ("dictionary", C.c_void_p),
                        ("release", C.CFUNCTYPE(None, C.POINTER(ArrowSchema))), ("private_data", C.c_void_p)]


class ArrowArray(C.Structure):
    pass


ArrowArray._fields_ = [("length", C.c_int64), ("null_count", C.c_int64), ("offset", C.c_int64), ("n_buffers", C.c_int64),
                       ("n_children", C.c_int64), ("buffers", C.POINTER(C.c_void_p)), ("children", C.c_void_p),
                       ("dictionary", C.c_void_p), ("release", C.CFUNCTYPE(None, C.POINTER(ArrowArray))),
                       ("private_data", C.c_void_p)]


class ArrowDeviceArray(C.Structure):
    _fields_ = [("array", ArrowArray), ("device_id", C.c_int64), ("device_type", C.c_int32), ("sync_event", C.c_void_p),
                ("reserved", C.c_int64 * 3)]


class ArrayView(C.Structure):  # ag_array_view
    _fields_ = [("type", C.c_int), ("length", C.c_int64), ("null_count", C.c_int64), ("offset", C.c_int64),
                ("validity", C.c_void_p), ("values", C.c_void_p), ("device_type", C.c_int32), ("device_id", C.c_int64)]


RELEASE_BUFFERS_FN = C.CFUNCTYPE(None, C.c_void_p)
DEVICE_CPU, DEVICE_CUDA, DEVICE_CUDA_HOST, DEVICE_CUDA_MANAGED = 1, 2, 3, 13

_SIGS.update({
    "ag_schema_format_to_type": [C.c_char_p, C.POINTER(_i)],
    "ag_device_array_describe": [C.POINTER(ArrowDeviceArray), C.POINTER(ArrowSchema), C.POINTER(ArrayView)],
    "ag_export_device_array": [_i, _i64, _i64, _i64, _p, _p, RELEASE_BUFFERS_FN, _p, _p, C.POINTER(ArrowDeviceArray), C.POINTER(ArrowSchema)],
    "ag_import_device_array": [C.POINTER(ArrowDeviceArray), C.POINTER(ArrowSchema), _p, C.POINTER(ArrayView)],
})

_SPECIAL = {
    "ag_type_to_schema_format": (C.c_char_p, [_i]),
    "ag_last_error": (None, [C.c_char_p, _sz]),
    "ag_version": (C.c_char_p, []),
    "ag_kernel_launch_count": (C.c_uint64, []),
}

_lib = None


def build(verbose=False):
    """Compile libarrowgpu.so (sm_100a kernels + C ABI) and libarrowgpu_host.so (C++ host mirror)
    in-tree.  nvcc cross-compiles without a GPU."""
    out = subprocess.run(["make", "-C", os.path.join(_HERE, "csrc"), "-j8"], capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError("libarrowgpu build failed:\n" + out.stdout[-4000:] + out.stderr[-4000:])
    if verbose:
        print(out.stdout[-2000:])
    out = subprocess.run(["make", "-C", os.path.join(_HERE, "host")], capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError("libarrowgpu_host build failed:\n" + out.stdout[-4000:] + out.stderr[-4000:])
    return LIB_PATH


def raw():
    """The CDLL itself (restype/argtypes set, no error translation)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeError(AG_ERR_CUDA, f"{LIB_PATH} is missing: run __graft_entry__.build() "
                              "(there is no CPU fallback)", "load")
        lib = C.CDLL(LIB_PATH)
        for name, argtypes in _SIGS.items():
            fn = getattr(lib, name)
            fn.restype = C.c_int
            fn.argtypes = argtypes
        for name, (restype, argtypes) in _SPECIAL.items():
            fn = getattr(lib, name)
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = lib
    return _lib


def last_error():
    buf = C.create_string_buffer(512)
    raw().ag_last_error(buf, 512)
    return buf.value.decode("utf-8", "replace")


def call(name, *args):
    """Call a status-returning entry point; raise NativeError on failure."""
    st = getattr(raw(), name)(*args)
    if st != AG_OK:
        raise NativeError(st, last_error(), name)
    return st


def call_status(name, *args):
    """Call and return (status, message) without raising."""
    st = getattr(raw(), name)(*args)
    return st, (last_error() if st != AG_OK else "")


def declared_symbols():
    """Every function name declared in include/arrowgpu.h and include/arrowgpu_cdata.h (for the export check)."""
    import re
    text = open(HEADER_PATH).read() + open(CDATA_HEADER_PATH).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ag_[a-z0-9_]+)\s*\(", text)))
