/*
 * arrowgpu.h — C ABI of the B200 (sm_100a) implementation of arrow-go's vectorised
 * columnar compute hot path.
 *
 * This header is the drop-in boundary: every entry point replaces one native
 * (c2goasm) inner loop or one pure-Go kernel body of the reference, and is what a
 * cgo package inside arrow-go would bind (see INTEGRATION.md for the Go side).
 * Reference citations are relative to the arrow-go tree (commit b3dacd2a).
 *
 * Conventions
 *   - Plain pointers and sizes only.  No CUDA or torch types appear here.
 *   - Every function returns an ag_status; AG_OK == 0.  ag_last_error() returns the
 *     calling thread's last message.  Status codes map 1:1 onto arrow-go's error
 *     sentinels (arrow/errors.go:21-28).
 *   - Two flavours of every compute entry point:
 *       ag_xxx(...)      HOST pointers.  Synchronous.  The library stages the
 *                        buffers to HBM (pinned, chunked, full-duplex), runs the
 *                        kernel(s) and copies the result back.  This is the form a
 *                        per-span exec.ArrayKernelExec binds.
 *       ag_xxx_dev(...)  DEVICE pointers + a stream.  Asynchronous.  Used when a
 *                        record batch has been uploaded once (ag_upload) and many
 *                        kernels run over it before anything is downloaded.
 *   - `type` arguments are arrow.Type ids (arrow/datatype.go:36-72 ==
 *     kernels/_lib/types.h:20-34); `op` arguments are kernels.ArithmeticOp values
 *     (arrow/compute/internal/kernels/base_arithmetic.go:37-82 ==
 *     _lib/base_arithmetic.cc:31-74).
 *   - Bitmaps are Arrow LSB-first bitmaps addressed by (byte pointer, bit offset).
 *     Bits outside [offset, offset+length) are never modified.
 *   - Value pointers only need element alignment (a slice start is only
 *     element-aligned); 16-byte aligned inputs take the vectorised path.
 *   - All entry points are thread-safe and re-entrant (cgo calls arrive on arbitrary
 *     OS threads, arrow/compute/exec.go:164-170).
 *   - There is NO CPU fallback: without a usable sm_100 device every compute entry
 *     point returns AG_ERR_CUDA.
 */
#ifndef ARROWGPU_H
#define ARROWGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes (arrow/errors.go:21-28) --------------------------------------- */
typedef int ag_status;
#define AG_OK                   0
#define AG_ERR_INVALID          1 /* arrow.ErrInvalid: overflow, divide by zero, length mismatch, bad argument */
#define AG_ERR_INDEX            2 /* arrow.ErrIndex: take index out of bounds */
#define AG_ERR_NOT_IMPLEMENTED  3 /* arrow.ErrNotImplemented */
#define AG_ERR_TYPE             4 /* arrow.ErrType */
#define AG_ERR_CUDA             5 /* device / driver failure (no sentinel in arrow-go; surfaces as ErrInvalid) */
#define AG_ERR_OOM              6 /* device or pinned allocation failed */

/* ---- arrow.Type ids that cross the boundary (arrow/datatype.go:36-72) ----------- */
#define AG_TYPE_NULL     0
#define AG_TYPE_BOOL     1
#define AG_TYPE_UINT8    2
#define AG_TYPE_INT8     3
#define AG_TYPE_UINT16   4
#define AG_TYPE_INT16    5
#define AG_TYPE_UINT32   6
#define AG_TYPE_INT32    7
#define AG_TYPE_UINT64   8
#define AG_TYPE_INT64    9
#define AG_TYPE_FLOAT16 10
#define AG_TYPE_FLOAT32 11
#define AG_TYPE_FLOAT64 12

/* ---- kernels.ArithmeticOp (base_arithmetic.go:37-82) ----------------------------- */
#define AG_OP_ADD             0
#define AG_OP_SUB             1
#define AG_OP_MUL             2
#define AG_OP_DIV             3
#define AG_OP_ABS             4
#define AG_OP_NEGATE          5
#define AG_OP_SIGN           20
#define AG_OP_ADD_CHECKED    21
#define AG_OP_SUB_CHECKED    22
#define AG_OP_MUL_CHECKED    23
#define AG_OP_DIV_CHECKED    24
#define AG_OP_ABS_CHECKED    25
#define AG_OP_NEGATE_CHECKED 26
/* Not ArithmeticOp values: the reference keeps these in separate enums (BitwiseOp scalar_arithmetic.go:183-189,
 * ShiftDir :286-291); one op space here so that they ride the same entry points.
 *   BIT_AND / BIT_OR / BIT_XOR: ag_arith_binary* on the integer types (every slot, like a3: bitwiseKernelOp :191-243
 *     runs the bitmap op over the value buffers); BIT_NOT: ag_arith_unary_same (bitwiseNot :257-259).
 *   SHIFT_*: ag_arith_checked* (ScalarBinaryNotNull slots).  An invalid amount (rhs < 0 or rhs >= bits for unsigned,
 *     rhs >= bits - 1 for SIGNED types — maxShift of shiftKernelSignedImpl :293-296) leaves lhs unchanged; the
 *     _CHECKED flavours also fail the call ("shift amount must be >= 0 and less than precision of type"). */
#define AG_OP_BIT_AND        64
#define AG_OP_BIT_OR         65
#define AG_OP_BIT_XOR        66
#define AG_OP_BIT_NOT        67
#define AG_OP_SHIFT_LEFT     68
#define AG_OP_SHIFT_RIGHT    69
#define AG_OP_SHIFT_LEFT_CHECKED  70
#define AG_OP_SHIFT_RIGHT_CHECKED 71

/* ---- kernels.CompareOperator (kernels/types.go:62-71) ---------------------------- */
#define AG_CMP_EQ 0
#define AG_CMP_NE 1
#define AG_CMP_GT 2
#define AG_CMP_GE 3
#define AG_CMP_LT 4 /* executed as GT with operands flipped, like scalar_compare.go:73-99 */
#define AG_CMP_LE 5 /* executed as GE with operands flipped */

/* operand shapes of the binary entry points (arr_arr / arr_scalar / scalar_arr) */
#define AG_SHAPE_AA 0
#define AG_SHAPE_AS 1
#define AG_SHAPE_SA 2

/* ---- bitmap binary ops (arrow/bitutil/bitmaps.go:601-639) ------------------------ */
#define AG_BITOP_AND     0
#define AG_BITOP_OR      1
#define AG_BITOP_XOR     2
#define AG_BITOP_ANDNOT  3 /* l & ~r */
#define AG_BITOP_XNOR    4
/* Kleene word ops (scalar_boolean.go:103-105,180-182,290-292) */
#define AG_KLEENE_AND     0
#define AG_KLEENE_OR      1
#define AG_KLEENE_ANDNOT  2

/* ---- kernels.NullSelectionBehavior (vector_selection.go:34-39) ------------------- */
#define AG_DROP_NULLS 0
#define AG_EMIT_NULLS 1

/* sentinel written to *first_bad / *bad_pos when no element failed */
#define AG_NO_ERROR_POS INT64_MAX

typedef void* ag_stream_t; /* opaque (a CUDA stream); NULL = the current device's default stream */
typedef void* ag_event_t;  /* opaque (a CUDA event) */
typedef void* ag_comm_t;   /* opaque: one rank of a multi-GPU communicator */

/* ================================================================================= *
 * Runtime, residency, streams
 * ================================================================================= */

/* Initialise one device and its stream pool.  The first call names the process DEFAULT device
 * (device < 0: LOCAL_RANK from the environment, else 0) — all a one-process-per-GPU rank needs.
 * Idempotent; every compute call initialises lazily with device -1 if this was never called.
 * A later ag_init(other) behaves like ag_set_device(other). */
ag_status ag_init(int device);
/* One process driving the whole box (the reference is ONE Go process whose take/filter fan out over
 * goroutines, arrow/compute/selection.go:127-150): initialise every visible device and enable peer
 * access between all pairs.  Then each worker thread picks its device with ag_set_device; streams,
 * pinned and device allocations, and NULL-stream calls follow the calling thread's current device,
 * and a call that is handed a stream always runs on that stream's device. */
ag_status ag_init_all(int* n_devices);
ag_status ag_set_device(int device);
ag_status ag_get_device(int* device);
ag_status ag_shutdown(void);
ag_status ag_device_count(int* count);
ag_status ag_device_info(int* device, int* sm_count, size_t* hbm_bytes, int* cc_major, int* cc_minor);
/* Copies the calling thread's last error message (NUL-terminated) into buf. */
void ag_last_error(char* buf, size_t buflen);
/* Library version string and the number of kernels this process has launched
 * (used by bench.py's gpu_launches and by the loaded-native-code check). */
const char* ag_version(void);
uint64_t ag_kernel_launch_count(void);

/* Pinned host memory: backs a Go memory.Allocator (arrow/memory/allocator.go:23-27);
 * shape follows arrow/memory/internal/cgoalloc/allocator.h:13-18.  64-byte aligned,
 * zero-initialised like memory.GoAllocator / mallocator (calloc). */
ag_status ag_host_alloc(void** ptr, size_t nbytes);
ag_status ag_host_realloc(void** ptr, size_t old_nbytes, size_t new_nbytes);
ag_status ag_host_free(void* ptr);
/* Page-lock memory the caller already owns (e.g. a Mallocator buffer). */
ag_status ag_host_register(void* ptr, size_t nbytes);
ag_status ag_host_unregister(void* ptr);

ag_status ag_dev_alloc(void** dptr, size_t nbytes);   /* stream-ordered pool, zero-filled */
ag_status ag_dev_free(void* dptr);
ag_status ag_dev_memset(void* dptr, int byte, size_t nbytes, ag_stream_t s);
ag_status ag_upload(void* dst_dev, const void* src_host, size_t nbytes, ag_stream_t s);
ag_status ag_download(void* dst_host, const void* src_dev, size_t nbytes, ag_stream_t s);
ag_status ag_copy_dev(void* dst_dev, const void* src_dev, size_t nbytes, ag_stream_t s);

ag_status ag_stream_create(ag_stream_t* s);
ag_status ag_stream_destroy(ag_stream_t s);
ag_status ag_stream_sync(ag_stream_t s);
ag_status ag_event_create(ag_event_t* e);
ag_status ag_event_destroy(ag_event_t e);
ag_status ag_event_record(ag_event_t e, ag_stream_t s);
ag_status ag_event_sync(ag_event_t e);
ag_status ag_event_elapsed_ms(ag_event_t start, ag_event_t stop, float* ms);
/* Writes `nbytes` of a scratch buffer (> L2) so the next timed launch starts cold. */
ag_status ag_flush_l2(ag_stream_t s);

/* ================================================================================= *
 * arrow/math Sum  — replaces sum_{float64,int64,uint64}_{avx2,sse4,neon}
 *   arrow/math/_lib/float64.c:20-26, int64.c:21-27, uint64.c; Go: float64.go:34-39.
 *   Validity is ignored (like the reference); n == 0 gives 0.
 *   Integer sums wrap (two's complement) — bit-exact for any order.
 *   Float64: default mode is a fixed-shape tree (result is a pure function of data
 *   and n, independent of grid/alignment; bit-exact with the reference whenever the
 *   sum is exactly representable, closer to the exact sum otherwise).
 *   ag_sum_f64_reforder reproduces the reference AVX2 association order
 *   (float64_avx2_amd64.s:36-43,86-164) bit-for-bit on any input.
 * ================================================================================= */
ag_status ag_sum_f64(const double* buf, size_t n, double* res);
ag_status ag_sum_i64(const int64_t* buf, size_t n, int64_t* res);
ag_status ag_sum_u64(const uint64_t* buf, size_t n, uint64_t* res);
ag_status ag_sum_f64_reforder(const double* buf, size_t n, double* res);
ag_status ag_sum_f64_dev(const double* d_buf, size_t n, double* d_res, ag_stream_t s);
ag_status ag_sum_i64_dev(const int64_t* d_buf, size_t n, int64_t* d_res, ag_stream_t s);
ag_status ag_sum_u64_dev(const uint64_t* d_buf, size_t n, uint64_t* d_res, ag_stream_t s);
ag_status ag_sum_f64_reforder_dev(const double* d_buf, size_t n, double* d_res, ag_stream_t s);

/* ================================================================================= *
 * Multi-GPU (SURVEY §8e): row-range shards, no data-path collective except the global Sum.
 *   Sharding rule: ag_shard_range — ceil-balanced, cuts at multiples of 64 rows (no two shards
 *   share a bitmap word).  Add / compare / filter / take run per shard with no exchange (take
 *   replicates `values`); a bounds / overflow error is the minimum of the shards' error words.
 *   Global Sum: ag_sum_*_global_dev runs the shard's reduction AND the fold over the ranks as
 *   one kernel — the final (sum, error) pair is stored into every rank's HBM mailbox over
 *   NVLink and folded in rank order, so every rank's *d_res holds the same bits, with no
 *   second launch and no host synchronisation.  Every rank of the communicator must make the
 *   call (in the same order when several are in flight).
 *   Setting up the mailboxes:
 *     one process per GPU : ag_comm_local_handle(world, h) on every rank; all-gather the
 *                           AG_COMM_HANDLE_BYTES handles with the caller's own plumbing (MPI,
 *                           torch.distributed, a socket); ag_comm_create(&c, world, rank, handles)
 *     one process, n GPUs : ag_init_all; ag_comm_create_local(comms, n, devices)
 *   NCCL (optional): ag_comm_unique_id on rank 0, broadcast the AG_COMM_ID_BYTES, then
 *   ag_comm_attach_nccl on every rank; ag_sum_i64_global_nccl_dev = per-GPU Sum followed by
 *   ncclAllReduce of the 8-byte result on the same stream.  libnccl.so.2 is dlopen'ed on
 *   first use (AG_ERR_NOT_IMPLEMENTED when the process has none).
 * ================================================================================= */
#define AG_COMM_HANDLE_BYTES 64
#define AG_COMM_ID_BYTES 128
ag_status ag_shard_range(int64_t n_rows, int shard, int n_shards, int64_t* start, int64_t* stop);
ag_status ag_comm_local_handle(int world, void* handle64);
ag_status ag_comm_create(ag_comm_t* comm, int world, int rank, const void* all_handles);
ag_status ag_comm_create_local(ag_comm_t* comms, int n, const int* devices);
ag_status ag_comm_unique_id(void* id128);
ag_status ag_comm_attach_nccl(ag_comm_t comm, const void* id128);
ag_status ag_comm_info(ag_comm_t comm, int* world, int* rank, int* device);
ag_status ag_comm_destroy(ag_comm_t comm);
ag_status ag_sum_i64_global_dev(ag_comm_t comm, const int64_t* d_buf, size_t n, int64_t* d_res, ag_stream_t s);
ag_status ag_sum_u64_global_dev(ag_comm_t comm, const uint64_t* d_buf, size_t n, uint64_t* d_res, ag_stream_t s);
ag_status ag_sum_f64_global_dev(ag_comm_t comm, const double* d_buf, size_t n, double* d_res, ag_stream_t s);
ag_status ag_sum_i64_global_nccl_dev(ag_comm_t comm, const int64_t* d_buf, size_t n, int64_t* d_res, ag_stream_t s);

/* ================================================================================= *
 * Integer min/max — replaces {int,uint}{8,16,32,64}_max_min_{avx2,sse4,neon}
 *   (internal/utils/_lib/min_max.c:23-125; Go: GetMinMaxInt8 ... GetMinMaxUint64,
 *   internal/utils/min_max.go) — the reduction behind Parquet column statistics
 *   (parquet/metadata/statistics_types.gen.go:160-190,464-490).  n == 0 gives the
 *   reference's initial values (type MAX, type MIN).  The device flavour writes
 *   {min, max} as two consecutive elements of the value type.
 * ================================================================================= */
ag_status ag_min_max(int type, const void* values, int64_t n, void* min_out, void* max_out);
ag_status ag_min_max_dev(int type, const void* d_values, int64_t n, void* d_min_max, ag_stream_t s);

/* ================================================================================= *
 * Arithmetic — replaces arithmetic_{binary,arr_scalar,scalar_arr,unary_same_types,
 *   unary_diff_type}_{avx2,sse4} (_lib/base_arithmetic.cc:465-483) and the pure-Go
 *   fallbacks of base_arithmetic.go.  Computed for EVERY slot (ScalarBinary
 *   semantics, helpers.go:193-236).  Ops: ADD/SUB/MUL (+_CHECKED aliases, which for
 *   these entry points are the unchecked loops exactly like the reference's native
 *   code: base_arithmetic.cc:445-462).  Integers wrap.  The scalar operand is a
 *   pointer to one element (host memory in both flavours).
 * ================================================================================= */
ag_status ag_arith_binary(int type, int8_t op, const void* l, const void* r, void* out, int64_t n);
ag_status ag_arith_arr_scalar(int type, int8_t op, const void* l, const void* scalar_r, void* out, int64_t n);
ag_status ag_arith_scalar_arr(int type, int8_t op, const void* scalar_l, const void* r, void* out, int64_t n);
ag_status ag_arith_unary_same(int type, int8_t op, const void* in, void* out, int64_t n);      /* ABS, NEGATE, SIGN (+_CHECKED aliases) */
ag_status ag_arith_unary_diff(int itype, int otype, int8_t op, const void* in, void* out, int64_t n); /* SIGN */
ag_status ag_arith_binary_dev(int type, int8_t op, int shape, const void* d_l, const void* d_r, void* d_out,
                              int64_t n, ag_stream_t s); /* scalar side: HOST pointer to one element */
/* Batched form for chunked arguments: ONE launch (device flavour) / one pipelined transfer
 * schedule (host flavour) for all the aligned spans iterateExecSpans yields for a call
 * (arrow/compute/executor.go:757-863).  A compute.Function that receives whole ChunkedDatums
 * (functions.go:30-41) binds this instead of a per-span kernel.  Results are identical to
 * calling ag_arith_binary[_dev] once per span.  For AS / SA shapes the scalar side of every
 * span must be the same host pointer to one element. */
typedef struct ag_span3 { const void* l; const void* r; void* out; int64_t n; } ag_span3;
ag_status ag_arith_binary_spans(int type, int8_t op, int shape, const ag_span3* spans, int64_t n_spans);
ag_status ag_arith_binary_spans_dev(int type, int8_t op, int shape, const ag_span3* spans, int64_t n_spans, ag_stream_t s);
ag_status ag_arith_unary_same_dev(int type, int8_t op, const void* d_in, void* d_out, int64_t n, ag_stream_t s);
ag_status ag_arith_unary_diff_dev(int itype, int otype, int8_t op, const void* d_in, void* d_out, int64_t n, ag_stream_t s);

/* Checked integer arithmetic with the reference's exact overflow predicate and slot
 * semantics — no native counterpart exists in the reference; this restates
 *   ADD_CHECKED / SUB_CHECKED: base_arithmetic.go:249-278 under ScalarBinaryNotNull
 *       (helpers.go:284-380): only slots valid in BOTH inputs are computed, null slots
 *       are written as 0;
 *   MUL_CHECKED: base_arithmetic.go:84-108,279-286 under ScalarBinary (all slots);
 *   DIV / DIV_CHECKED: base_arithmetic.go:154-161,287-294 (divide by zero -> error),
 *       ScalarBinaryNotNull.
 * lvalid / rvalid may be NULL (= all valid); offsets are bit offsets.  A NULL scalar
 * operand pointer means a null scalar (whole output untouched, status OK).
 * On overflow / divide by zero returns AG_ERR_INVALID and *first_bad (may be NULL)
 * receives the lowest failing row; otherwise AG_NO_ERROR_POS. */
ag_status ag_arith_checked(int type, int8_t op, int shape,
                           const void* l, const uint8_t* lvalid, int64_t loff,
                           const void* r, const uint8_t* rvalid, int64_t roff,
                           void* out, int64_t n, int64_t* first_bad);
/* abs / negate (checked) on signed integers: AbsoluteValueChecked / NegateChecked,
 * base_arithmetic.go:295-340 under ScalarUnary (EVERY slot, null or not): a slot equal to
 * MinInt gives AG_ERR_INVALID "overflow"; other slots as the unchecked kernels.  Unsigned and
 * floating types never fail (they behave like ag_arith_unary_same). */
ag_status ag_arith_unary_checked(int type, int8_t op, const void* in, void* out, int64_t n, int64_t* first_bad);
ag_status ag_arith_unary_checked_dev(int type, int8_t op, const void* d_in, void* d_out, int64_t n, int64_t* d_first_bad, ag_stream_t s);
/* Device flavour: *d_first_bad must be initialised to AG_NO_ERROR_POS by the caller
 * (ag_dev_memset is not enough: use ag_error_word_reset_dev); it is only lowered. */
ag_status ag_arith_checked_dev(int type, int8_t op, int shape,
                               const void* d_l, const uint8_t* d_lvalid, int64_t loff,
                               const void* d_r, const uint8_t* d_rvalid, int64_t roff,
                               void* d_out, int64_t n, int64_t* d_first_bad, ag_stream_t s);
ag_status ag_error_word_reset_dev(int64_t* d_word, ag_stream_t s);

/* ================================================================================= *
 * Numeric casts — replaces cast_type_numeric_{avx2,sse4} (_lib/cast_numeric.cc:22-101, Go
 *   dispatch cast_numeric.go:101-131) for the 10 numeric types, and the checks of
 *   numeric_cast.go that frame it under safe CastOptions (what implicit promotion uses:
 *   compute/exec.go:101-121 -> CastDatum(SafeCastOptions)):
 *     int -> int    intsCanFit/intsInRange (helpers.go:545-653), skipped when AllowIntOverflow
 *     int -> float  checkIntToFloatTrunc   (numeric_cast.go:698-729): |v| <= 2^24 / 2^53
 *     float -> int  checkFloatTrunc        (numeric_cast.go:613-660): OutT(v) converted back != v
 *   the last two skipped when AllowFloatTruncate.  Every slot is converted (nulls too, like
 *   castNumberToNumberUnsafe, helpers.go:690-703); the checks look only at valid slots.
 *   Bit-exact with the reference loops for every input whose converted value is representable
 *   in the output type; out-of-range float -> int is not defined by the reference (its AVX2 body,
 *   SSE4 body and scalar tail disagree) — here: 64-bit truncation (NaN/overflow -> INT64_MIN)
 *   then wrap to the output width, the pure-Go amd64 behaviour.
 *   Checked flavour: AG_ERR_INVALID + lowest failing row in *first_bad (else AG_NO_ERROR_POS).
 * ================================================================================= */
ag_status ag_cast_numeric(int itype, int otype, const void* in, void* out, int64_t n);
ag_status ag_cast_numeric_dev(int itype, int otype, const void* d_in, void* d_out, int64_t n, ag_stream_t s);
ag_status ag_cast_numeric_checked(int itype, int otype, const void* in, const uint8_t* valid, int64_t valid_offset,
                                  void* out, int64_t n, int allow_int_overflow, int allow_float_truncate, int64_t* first_bad);
/* *d_first_bad must hold AG_NO_ERROR_POS (ag_error_word_reset_dev); it is only lowered. */
ag_status ag_cast_numeric_checked_dev(int itype, int otype, const void* d_in, const uint8_t* d_valid, int64_t valid_offset,
                                      void* d_out, int64_t n, int allow_int_overflow, int allow_float_truncate,
                                      int64_t* d_first_bad, ag_stream_t s);

/* ================================================================================= *
 * cumulative_sum / cumulative_sum_checked — replaces cumulativeSum{NoNulls,WithNulls}[Checked]
 *   (arrow/compute/internal/kernels/vector_cumulative.go:228-330; options CumulativeOptions
 *   {Start, SkipNulls} :92-99; chunked input = one logical sequence, :385-410).
 *   out[i] = start + sum of the valid in[j], j <= i.  Null input slot -> null output slot (value 0).
 *   Without skip_nulls every slot after the first null is null too and nothing accumulates past
 *   it.  `checked`: AG_ERR_INVALID "overflow" at the first running sum outside the type's range
 *   (integers only; floats never fail), lowest failing row in *first_bad.
 *   Integers: bit-exact.  Floats: single-pass parallel scan with a fixed (data- and n-determined)
 *   association — bit-exact with the reference's left-to-right loop whenever every partial sum
 *   is exactly representable, otherwise within the usual summation error bound (DESIGN.md).
 *
 *   Device flavour: the running value and the encountered-null flag live in a 32-byte device
 *   block (ag_cumsum_state) so that the chunks of a chunked column are a chain of launches on
 *   one stream; initialise it with ag_cumulative_sum_state_init_dev (start_host: pointer to one
 *   element of `type`, or NULL for zero).  d_out_valid (bit offset out_valid_offset) is required
 *   when d_valid is given and otherwise optional (pass it for every chunk when any chunk has
 *   nulls); state.null_count accumulates the null slots written.
 * ================================================================================= */
typedef struct ag_cumsum_state { uint64_t lo; int64_t hi; int64_t encountered_null; int64_t null_count; } ag_cumsum_state;
ag_status ag_cumulative_sum(int type, const void* in, const uint8_t* valid, int64_t valid_offset, int64_t n,
                            const void* start, int skip_nulls, int checked,
                            void* out, uint8_t* out_valid, int64_t* null_count, int64_t* first_bad);
ag_status ag_cumulative_sum_state_init_dev(void* d_state, int type, const void* start_host, ag_stream_t s);
ag_status ag_cumulative_sum_dev(int type, const void* d_in, const uint8_t* d_valid, int64_t valid_offset, int64_t n,
                                int skip_nulls, int checked, void* d_out, uint8_t* d_out_valid, int64_t out_valid_offset,
                                void* d_state, int64_t* d_first_bad, ag_stream_t s);

/* ================================================================================= *
 * Comparisons -> bitmap — replaces comparison_{equal,not_equal,greater,greater_equal}
 *   _{arr_arr,arr_scalar,scalar_arr}_{avx2,sse4} (_lib/scalar_comparison.cc:210-256)
 *   and compareKernel (scalar_comparisons.go:199-218).  `out_bits` points at the byte
 *   holding the first output bit, `bit_offset` is used mod 8 exactly like the
 *   reference; bits outside the written range are preserved.  LT/LE are accepted and
 *   executed by operand flipping.  NaN: every predicate false except NE.
 * ================================================================================= */
ag_status ag_compare(int type, int cmp, int shape, const void* l, const void* r,
                     uint8_t* out_bits, int64_t n, int bit_offset);
ag_status ag_compare_dev(int type, int cmp, int shape, const void* d_l, const void* d_r,
                         uint8_t* d_out_bits, int64_t n, int bit_offset, ag_stream_t s);
/* Named forms with the reference's exact native signature (type,l,r,out,length,offset). */
ag_status ag_cmp_eq_aa(int type, const void* l, const void* r, void* out, int64_t n, int offset);
ag_status ag_cmp_eq_as(int type, const void* l, const void* r, void* out, int64_t n, int offset);
ag_status ag_cmp_eq_sa(int type, const void* l, const void* r, void* out, int64_t n, int offset);
ag_status ag_cmp_ne_aa(int type, const void* l, const void* r, void* out, int64_t n, int offset);
ag_status ag_cmp_ne_as(int type, const void* l, const void* r, void* out, int64_t n, int offset);
ag_status ag_cmp_ne_sa(int type, const void* l, const void* r, void* out, int64_t n, int offset);
ag_status ag_cmp_gt_aa(int type, const void* l, const void* r, void* out, int64_t n, int offset);
ag_status ag_cmp_gt_as(int type, const void* l, const void* r, void* out, int64_t n, int offset);
ag_status ag_cmp_gt_sa(int type, const void* l, const void* r, void* out, int64_t n, int offset);
ag_status ag_cmp_ge_aa(int type, const void* l, const void* r, void* out, int64_t n, int offset);
ag_status ag_cmp_ge_as(int type, const void* l, const void* r, void* out, int64_t n, int offset);
ag_status ag_cmp_ge_sa(int type, const void* l, const void* r, void* out, int64_t n, int offset);

/* ================================================================================= *
 * Bitmaps — replaces bitmap_aligned_{and,or,and_not,xor}_{avx2,sse4}
 *   (arrow/bitutil/_lib/bitmap_ops.c:24-46) plus the Go paths around them:
 *   alignedBitmapOp / unalignedBitmapOp (bitmaps.go:527-591), CopyBitmap /
 *   InvertBitmap (:483-491), SetBitsTo (bitutil.go:158), CountSetBits (:89).
 *   Arbitrary bit offsets on every operand; `out` may alias an input with the same
 *   offset (propagateNulls accumulates in place, executor.go:340-347).
 * ================================================================================= */
ag_status ag_bitmap_op(int bitop, const uint8_t* l, int64_t loff, const uint8_t* r, int64_t roff,
                       uint8_t* out, int64_t ooff, int64_t nbits);
ag_status ag_bitmap_copy(const uint8_t* src, int64_t soff, int64_t nbits, uint8_t* dst, int64_t doff);
ag_status ag_bitmap_invert(const uint8_t* src, int64_t soff, int64_t nbits, uint8_t* dst, int64_t doff);
ag_status ag_bitmap_set(uint8_t* bits, int64_t off, int64_t nbits, int value);
ag_status ag_bitmap_popcount(const uint8_t* bits, int64_t off, int64_t nbits, int64_t* count);
ag_status ag_bitmap_op_dev(int bitop, const uint8_t* d_l, int64_t loff, const uint8_t* d_r, int64_t roff,
                           uint8_t* d_out, int64_t ooff, int64_t nbits, ag_stream_t s);
ag_status ag_bitmap_copy_dev(const uint8_t* d_src, int64_t soff, int64_t nbits, uint8_t* d_dst, int64_t doff, ag_stream_t s);
ag_status ag_bitmap_invert_dev(const uint8_t* d_src, int64_t soff, int64_t nbits, uint8_t* d_dst, int64_t doff, ag_stream_t s);
ag_status ag_bitmap_set_dev(uint8_t* d_bits, int64_t off, int64_t nbits, int value, ag_stream_t s);
/* *d_count is overwritten with the population count of [off, off+nbits). */
ag_status ag_bitmap_popcount_dev(const uint8_t* d_bits, int64_t off, int64_t nbits, int64_t* d_count, ag_stream_t s);

/* Kleene logic on (validity, data) pairs — computeKleene, scalar_boolean.go:29-65 with
 * the word lambdas at :103-105 (and), :180-182 (or), :290-292 (and_not).  lvalid /
 * rvalid may be NULL (= all valid).  Both outputs use bit offset ooff. */
ag_status ag_kleene(int kop, const uint8_t* lvalid, const uint8_t* ldata, int64_t loff,
                    const uint8_t* rvalid, const uint8_t* rdata, int64_t roff,
                    uint8_t* out_valid, uint8_t* out_data, int64_t ooff, int64_t nbits);
ag_status ag_kleene_dev(int kop, const uint8_t* d_lvalid, const uint8_t* d_ldata, int64_t loff,
                        const uint8_t* d_rvalid, const uint8_t* d_rdata, int64_t roff,
                        uint8_t* d_out_valid, uint8_t* d_out_data, int64_t ooff, int64_t nbits, ag_stream_t s);

/* ================================================================================= *
 * Filter — replaces PrimitiveFilter (vector_selection.go:449-520) =
 *   getFilterOutputSize (:57-81) + primitiveFilterImpl (:267-395) + filterWriter
 *   (:397-421), and GetTakeIndices (:102-236).
 *   values: fixed width, bit_width in {8,16,32,64}; `vals` points at element 0 of the
 *   buffer and voff is the element offset (needed for the validity bitmap too).
 *   vvalid / mvalid may be NULL.  Output: stable compaction; out_valid (may be NULL when the
 *   output cannot contain nulls) receives the compacted validity starting at bit 0;
 *   EMIT_NULLS writes value 0 / validity 0 for null mask slots.
 * ================================================================================= */
ag_status ag_filter_output_size(const uint8_t* mask, const uint8_t* mvalid, int64_t moff, int64_t n,
                                int null_selection, int64_t* out_len);
ag_status ag_filter_primitive(int bit_width, const void* vals, const uint8_t* vvalid, int64_t voff,
                              const uint8_t* mask, const uint8_t* mvalid, int64_t moff, int64_t n,
                              int null_selection, void* out, uint8_t* out_valid,
                              int64_t* out_len, int64_t* out_nulls);
ag_status ag_filter_output_size_dev(const uint8_t* d_mask, const uint8_t* d_mvalid, int64_t moff, int64_t n,
                                    int null_selection, int64_t* d_out_len, ag_stream_t s);
/* out_capacity = number of rows d_out (and d_out_valid) can hold: the exact output length
 * when the caller ran ag_filter_output_size_dev first, or n as an upper bound.  Rows past the
 * capacity are dropped; *d_out_len always receives the full number of emitted rows so a
 * truncation is detectable.  d_out_valid (may be NULL when the output cannot contain nulls:
 * no values validity, and DROP_NULLS or no mask validity) must be 4-byte aligned and hold
 * ceil(out_capacity/32) 32-bit words; it is fully overwritten (Arrow buffers are padded to 64 B). */
ag_status ag_filter_primitive_dev(int bit_width, const void* d_vals, const uint8_t* d_vvalid, int64_t voff,
                                  const uint8_t* d_mask, const uint8_t* d_mvalid, int64_t moff, int64_t n,
                                  int null_selection, void* d_out, uint8_t* d_out_valid, int64_t out_capacity,
                                  int64_t* d_out_len, ag_stream_t s);
/* Fused Greater/…(values, scalar) + Filter: one pass over `values`, no intermediate
 * mask (SURVEY §8d: 8 + 8s bytes/row).  Not a reference entry point — an optimisation
 * the plugin applies to the greater→filter pipeline of config 3; results are identical
 * to ag_compare followed by ag_filter_primitive. */
ag_status ag_filter_compare_scalar_dev(int type, int cmp, const void* d_vals, const void* scalar_host,
                                       int64_t n, void* d_out, int64_t out_capacity, int64_t* d_out_len, ag_stream_t s);
/* GetTakeIndices: mask -> row indices; index_width 16 or 32 bits (the reference picks
 * uint16 when n < 65535 else uint32, vector_selection.go:229-235). */
ag_status ag_take_indices(int index_width, const uint8_t* mask, const uint8_t* mvalid, int64_t moff, int64_t n,
                          int null_selection, void* out_idx, uint8_t* out_valid, int64_t* out_len);
ag_status ag_take_indices_dev(int index_width, const uint8_t* d_mask, const uint8_t* d_mvalid, int64_t moff, int64_t n,
                              int null_selection, void* d_out_idx, uint8_t* d_out_valid, int64_t out_capacity,
                              int64_t* d_out_len, ag_stream_t s);

/* ================================================================================= *
 * Take — replaces PrimitiveTake (vector_selection.go:1162-1192) = checkIndexBounds
 *   (helpers.go:929-981) + primitiveTakeImpl (:813-988).
 *   out[i] = values[voff + idx[i]]; out_valid[i] = ivalid[ioff+i] & vvalid[voff+idx[i]].
 *   Null output slots carry value 0 (the reference leaves its zero-initialised
 *   allocation untouched).  idx_width in {8,16,32,64}; idx_signed: indices are
 *   reinterpreted as unsigned after the bounds check (:1147-1159).  With bounds_check,
 *   an out-of-range VALID index gives AG_ERR_INDEX, *bad_pos = lowest offending row and
 *   *bad_index = its value ("%d out of bounds", helpers.go:951).
 * ================================================================================= */
ag_status ag_take_primitive(int bit_width, const void* vals, const uint8_t* vvalid, int64_t voff, int64_t vlen,
                            int idx_width, int idx_signed, const void* idx, const uint8_t* ivalid, int64_t ioff,
                            int64_t n, int bounds_check, void* out, uint8_t* out_valid,
                            int64_t* out_nulls, int64_t* bad_pos, int64_t* bad_index);
/* d_out_valid: 4-byte aligned, offset 0.  *d_bad_pos must have been reset with
 * ag_error_word_reset_dev and is only lowered. */
ag_status ag_take_primitive_dev(int bit_width, const void* d_vals, const uint8_t* d_vvalid, int64_t voff, int64_t vlen,
                                int idx_width, int idx_signed, const void* d_idx, const uint8_t* d_ivalid, int64_t ioff,
                                int64_t n, int bounds_check, void* d_out, uint8_t* d_out_valid,
                                int64_t* d_bad_pos, ag_stream_t s);
/* Routing of large takes (results never depend on it).  Random indices into a values table far larger
 * than L2 go through the windowed path (partition indices by 16 MB table window -> gather window by
 * window out of L2 -> un-permute); sorted / clustered indices and small calls use the direct gather
 * (the reference switches loop shape the same way, vector_selection.go:897-911).
 * mode: 0 automatic (default), 1 always direct, 2 windowed whenever the shapes allow it.
 * min_rows / min_table_bytes / window_bytes: thresholds of the automatic mode and the window size;
 * values <= 0 keep the current setting.  Process-wide. */
ag_status ag_take_set_policy(int mode, int64_t min_rows, int64_t min_table_bytes, int64_t window_bytes);

/* ================================================================================= *
 * is_in / unique for fixed-width values of 1/2/4/8 bytes (SURVEY 8f rank 3) — the memo-table kernels of
 *   kernels/scalar_set_lookup.go:112-413 and kernels/vector_hash.go.  Values are compared by their RAW
 *   BYTES like the reference's memo tables (floats: NaN == NaN of the same payload, -0.0 != +0.0).
 *   is_in: out_data / out_valid are bitmaps at bit offset 0 (4-byte aligned); per row
 *     valid value: in the set -> (true, valid); else INCONCLUSIVE and the set holds a null -> (false, null);
 *                  else (false, valid)
 *     null       : MATCH and the set holds a null -> (true, valid); SKIP, or MATCH without one -> (false, valid);
 *                  else (false, null)                                   (isInKernelExec :373-413)
 *   unique: the distinct values in order of first appearance, a null kept once where it first appears;
 *     *out_len receives the count (capacity n is always enough).
 *   `offset` / `set_offset` are element offsets into both the values buffer and the validity bitmap.
 * ================================================================================= */
#define AG_NULL_MATCH        0
#define AG_NULL_SKIP         1
#define AG_NULL_EMIT_NULL    2
#define AG_NULL_INCONCLUSIVE 3
ag_status ag_is_in(int bit_width, const void* vals, const uint8_t* valid, int64_t offset, int64_t n,
                   const void* set_vals, const uint8_t* set_valid, int64_t set_offset, int64_t set_n, int null_behavior,
                   uint8_t* out_data, uint8_t* out_valid, int64_t* out_nulls);
ag_status ag_is_in_dev(int bit_width, const void* d_vals, const uint8_t* d_valid, int64_t offset, int64_t n,
                       const void* d_set_vals, const uint8_t* d_set_valid, int64_t set_offset, int64_t set_n, int null_behavior,
                       uint8_t* d_out_data, uint8_t* d_out_valid, int64_t* d_null_count, ag_stream_t s);
ag_status ag_unique(int bit_width, const void* vals, const uint8_t* valid, int64_t offset, int64_t n,
                    void* out, uint8_t* out_valid, int64_t* out_len, int64_t* out_nulls);
ag_status ag_unique_dev(int bit_width, const void* d_vals, const uint8_t* d_valid, int64_t offset, int64_t n,
                        void* d_out, uint8_t* d_out_valid, int64_t capacity, int64_t* d_out_len, ag_stream_t s);
/* unique's table policy: a column of more than `small_rows` rows (default 2^21) is first inserted into a table of
 * `small_slots` slots (a power of two, default 2^22 = 64 MB, L2-resident); the full-size table (2n slots) is filled only
 * when more than small_slots/2 distinct values turn up — decided on the device, never changes a result.  0 = default. */
ag_status ag_unique_set_policy(int64_t small_rows, int64_t small_slots);

/* ================================================================================= *
 * dictionary_encode for fixed-width values of 1/2/4/8 bytes — kernels/vector_hash.go:83-141
 *   (NullEncodingBehavior, DictionaryEncodeOptions), :144-241 (dictionaryEncodeAction), :359-385
 *   (doAppendNumeric), :854-872 (dictionaryEncodeFinalize).  Same key equality and table policy as unique
 *   (raw bytes; ag_unique_set_policy).
 *   dict: the distinct values in order of first appearance; indices: one int32 per row = its value's position.
 *   AG_NULL_ENCODING_MASK  : a null row gets index 0 and a null in the indices (indices_valid, bit offset 0);
 *                            the dictionary has no null entry.
 *   AG_NULL_ENCODING_ENCODE: the nulls share one dictionary entry placed where the first null appears (its
 *                            dict_valid bit cleared, its value bytes 0); the indices have no nulls.
 *   Any other null_encoding is AG_ERR_INVALID.  An input with a validity bitmap needs indices_valid in mask mode
 *   and dict_valid in encode mode.  indices / indices_valid / dict_valid: 4-byte aligned, bit offset 0; a given
 *   indices_valid is fully written (ceil(n/32) words).  `offset` is the element offset into both the values
 *   buffer and the validity bitmap.  n < 2^31 rows per call.
 *   Host flavour: dict (and dict_valid) need room for n entries; *dict_len / *index_nulls receive the counts.
 *   Device flavour: d_counts[0] = dictionary length, d_counts[1] = null count of the indices; entries past
 *   dict_capacity are dropped (d_counts[0] still receives the full length, so a truncation is detectable).
 * ================================================================================= */
#define AG_NULL_ENCODING_MASK   0
#define AG_NULL_ENCODING_ENCODE 1
ag_status ag_dictionary_encode(int bit_width, const void* vals, const uint8_t* valid, int64_t offset, int64_t n,
                               int null_encoding, int32_t* indices, uint8_t* indices_valid, void* dict,
                               uint8_t* dict_valid, int64_t* dict_len, int64_t* index_nulls);
ag_status ag_dictionary_encode_dev(int bit_width, const void* d_vals, const uint8_t* d_valid, int64_t offset, int64_t n,
                                   int null_encoding, int32_t* d_indices, uint8_t* d_indices_valid, void* d_dict,
                                   uint8_t* d_dict_valid, int64_t dict_capacity, int64_t* d_counts, ag_stream_t s);

/* ================================================================================= *
 * sort_indices, one fixed-width column (SURVEY 8f rank 3) — replaces kernels.SortIndices for a single
 *   key (vector_sort.go:385-481, vector_sort_internal.go:36-150,250-300): a STABLE permutation of
 *   0..n-1 as uint64 row indices,
 *     null_placement 0 (NullsAtEnd)  : [finite in key order | NaN in row order | null in row order]
 *     null_placement 1 (NullsAtStart): [null in row order | NaN in row order | finite in key order]
 *   order 0 ascending / 1 descending (ties keep row order either way; -0.0 == +0.0).
 *   `offset` is the slice's element offset into both the values buffer and the validity bitmap.
 *   The device flavour synchronises the stream once (a 2 KB histogram read-back decides which radix
 *   passes can be skipped).  n < 2^32 rows per call.
 * ================================================================================= */
ag_status ag_sort_indices(int type, const void* vals, const uint8_t* valid, int64_t offset, int64_t n, int order,
                          int null_placement, uint64_t* out_indices, int64_t* null_count, int64_t* nan_count);
ag_status ag_sort_indices_dev(int type, const void* d_vals, const uint8_t* d_valid, int64_t offset, int64_t n, int order,
                              int null_placement, uint64_t* d_out_indices, int64_t* null_count, int64_t* nan_count, ag_stream_t s);

/* ================================================================================= *
 * Parquet decode primitives (SURVEY 8f rank 4: the feeder side) — the SIMD leaf loops arrow-go links under
 *   parquet/internal, so pages can be decoded into device-resident Arrow buffers.
 *   ag_parquet_unpack32 ↔ unpack32_avx2 (parquet/internal/utils/_lib/bit_packing_avx2.c:1772): values of
 *     num_bits (0..32) bits, LSB-first, 32 per group -> uint32; only whole groups are unpacked
 *     (batch_size/32*32, returned in *unpacked) — the caller handles the tail like BitReader.GetBatch.
 *     d_in 4-byte aligned, d_out 16-byte aligned.
 *   ag_parquet_bytes_to_bools ↔ bytes_to_bools (utils/_lib/unpack_bool.c:21): bit j of byte i -> out[8i+j] (0/1).
 *   ag_parquet_def_levels_to_bitmap ↔ DefLevelsToBitmap (parquet/file/level_conversion.go:134-184 over
 *     levels_to_bitmap / extract_bits, bmi/_lib/bitmap_bmi2.c:24-47): appends validity bits at
 *     valid_bits_offset.  repeated_ancestor_def_level < 0: no repeated parent — bit i = def[i] >= def_level,
 *     values_read = n (error if n > read_upper_bound).  Otherwise only slots with def >= the ancestor level
 *     produce a bit.  *null_count is INCREMENTED by values_read - set bits (like the reference); the device
 *     flavour returns {values_read, set bits} in d_counts[2].  n == 0 leaves valid_bits untouched.
 * ================================================================================= */
ag_status ag_parquet_unpack32(const uint32_t* in, uint32_t* out, int64_t batch_size, int num_bits, int64_t* unpacked);
ag_status ag_parquet_unpack32_dev(const uint32_t* d_in, uint32_t* d_out, int64_t batch_size, int num_bits, int64_t* unpacked, ag_stream_t s);
ag_status ag_parquet_bytes_to_bools(const uint8_t* bytes, int64_t len, uint8_t* out, int64_t outlen);
ag_status ag_parquet_bytes_to_bools_dev(const uint8_t* d_bytes, int64_t len, uint8_t* d_out, int64_t outlen, ag_stream_t s);
ag_status ag_parquet_def_levels_to_bitmap(const int16_t* def_levels, int64_t n, int def_level, int repeated_ancestor_def_level,
                                          uint8_t* valid_bits, int64_t valid_bits_offset, int64_t read_upper_bound,
                                          int64_t* values_read, int64_t* null_count);
ag_status ag_parquet_def_levels_to_bitmap_dev(const int16_t* d_def_levels, int64_t n, int def_level, int repeated_ancestor_def_level,
                                              uint8_t* d_valid_bits, int64_t valid_bits_offset, int64_t read_upper_bound,
                                              int64_t* d_counts, ag_stream_t s);

/* ================================================================================= *
 * Parity helpers for inputs too large to bring back to the host (SURVEY §8d):
 * order-sensitive 64-bit checksum  sum_i mix64(i) * word_i  (mod 2^64)  over a buffer
 * viewed as little-endian uint64 words (n_words = nbytes/8), and a counter-based
 * generator so 1B-row datasets are produced on the device and reproduced on the CPU.
 * ================================================================================= */
ag_status ag_checksum64_dev(const void* d_buf, size_t n_words, uint64_t* d_res, ag_stream_t s);
/* kind: 0 = splitmix64(seed + i) as u64; 1 = uniform int64 in [lo, hi] (hi-lo+1 <= 2^32, via
 * multiply-shift on the high 32 bits); 2 = uniform int32 in [lo, hi]; 3 = double(k) with k
 * uniform integer in [lo, hi]; 4 = bitmap with P(bit)=lo/hi (n = bits); 5 / 6 = sorted / reverse-sorted int32
 * ramp over [lo, hi] (the sorted index datasets of SURVEY §8d). */
ag_status ag_generate_dev(int kind, uint64_t seed, int64_t lo, int64_t hi, void* d_out, size_t n, ag_stream_t s);

#ifdef __cplusplus
}
#endif
#endif /* ARROWGPU_H */
