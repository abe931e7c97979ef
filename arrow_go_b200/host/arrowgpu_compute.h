// arrowgpu_compute.h — host-side mirror of arrow-go's compute interface for the hot path,
// written in C++ because no Go toolchain exists in the build image (see DESIGN.md §boundary).
//
// Same names, argument meaning and error behaviour as the reference (paths relative to the
// arrow-go tree, commit b3dacd2a):
//   exec::ArraySpan / ExecSpan / ExecResult / KernelCtx / ScalarKernel / VectorKernel
//                                   arrow/compute/exec/{span.go:76-88,548-576, kernel.go:457-727}
//   compute::Datum / Function / FunctionRegistry / ExecCtx / CallFunction
//                                   arrow/compute/{datum.go, functions.go:30-41, registry.go:30-133,
//                                   executor.go:46-122, exec.go:59-193}
//   compute::Add/Subtract/Multiply/…  arrow/compute/arithmetic.go:1090-1142
//   compute::Filter / Take            arrow/compute/selection.go:304,657
//   math::Float64Funcs::Sum …         arrow/math/float64.go:34-39
//
// B200-first difference: buffers live in HBM.  An Array is uploaded once (Array::FromHost —
// "DMA once per record batch"), every kernel runs on device-resident spans through the *_dev
// entry points of include/arrowgpu.h, and results are downloaded only when asked (ToHost).
// There is no CPU execution path in this layer.
#pragma once

#include <stdint.h>
#include <functional>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../include/arrowgpu.h"
#include "../../include/arrowgpu_cdata.h"

namespace arrowgpu {

// ---- arrow.Type (arrow/datatype.go:36-72) -----------------------------------------------
enum class Type : int {
  NA = 0, BOOL = 1, UINT8 = 2, INT8 = 3, UINT16 = 4, INT16 = 5, UINT32 = 6, INT32 = 7,
  UINT64 = 8, INT64 = 9, FLOAT16 = 10, FLOAT32 = 11, FLOAT64 = 12,
  DICTIONARY = 29  // int32 indices + a dictionary of the value type (dictionary_encode's output)
};
int BitWidth(Type t);  // 1 for BOOL; 0 for DICTIONARY: no kernel may take a dictionary array for its int32 indices
const char* TypeName(Type t);
bool IsInteger(Type t);
bool IsSignedInteger(Type t);
bool IsFloating(Type t);
bool IsNumeric(Type t);

constexpr int64_t kUnknownNullCount = -1;  // array.UnknownNullCount

// ---- errors (arrow/errors.go:21-28) -------------------------------------------------------
struct Status {
  int code = AG_OK;  // AG_ERR_INVALID == arrow.ErrInvalid, AG_ERR_INDEX == arrow.ErrIndex, ...
  std::string msg;
  bool ok() const { return code == AG_OK; }
  static Status OK() { return Status(); }
  static Status Make(int c, std::string m) { Status s; s.code = c; s.msg = std::move(m); return s; }
  static Status Invalid(std::string m) { return Make(AG_ERR_INVALID, std::move(m)); }
  static Status NotImplemented(std::string m) { return Make(AG_ERR_NOT_IMPLEMENTED, std::move(m)); }
  static Status TypeError(std::string m) { return Make(AG_ERR_TYPE, std::move(m)); }
  static Status IndexError(std::string m) { return Make(AG_ERR_INDEX, std::move(m)); }
  static Status FromNative(int c);  // appends ag_last_error()
};

// ---- memory: device-resident buffers (memory.Buffer analogue) -------------------------------
class Buffer {
 public:
  ~Buffer();
  uint8_t* data() const { return data_; }
  int64_t size() const { return size_; }
  static Status Allocate(int64_t nbytes, std::shared_ptr<Buffer>* out);          // zero-filled, 64-B padded
  static Status FromHost(const void* host, int64_t nbytes, std::shared_ptr<Buffer>* out);
  // Foreign device memory (an imported ArrowDeviceArray): not freed, `on_release` runs when the last
  // reference goes away (memory.Buffer with a custom release, arrow/cdata/cdata.go importedBuffer).
  static std::shared_ptr<Buffer> Wrap(const void* device_ptr, int64_t nbytes, std::function<void()> on_release);
  Status ToHost(void* host, int64_t nbytes, int64_t byte_offset = 0) const;
 private:
  uint8_t* data_ = nullptr;
  int64_t size_ = 0;
  bool foreign_ = false;
  std::function<void()> on_release_;
};

// arrow.ArrayData for primitive / boolean / dictionary arrays (arrow/array/data.go:30-42)
struct ArrayData {
  Type type = Type::NA;
  int64_t length = 0;
  int64_t null_count = 0;  // kUnknownNullCount allowed
  int64_t offset = 0;
  std::shared_ptr<Buffer> buffers[2];  // [0] validity bitmap (may be null), [1] values / boolean data (DICTIONARY: int32 indices)
  std::shared_ptr<ArrayData> dictionary;  // DICTIONARY only: the values the indices point at (its type is the value type)
  std::shared_ptr<ArrayData> Slice(int64_t off, int64_t len) const;  // array.NewSlice semantics
  // validity (LSB-first bitmap, `offset` applies) may be NULL; values must hold (offset+length) elements
  static Status FromHost(Type type, int64_t length, int64_t offset, const uint8_t* validity, const void* values,
                         int64_t null_count, std::shared_ptr<ArrayData>* out);
  // Copies the logical [0,length) range out: values (length elements, or ceil(length/8) bytes for BOOL,
  // bit 0 = element 0; the int32 indices for DICTIONARY) and validity (ceil(length/8) bytes; all ones when there is no bitmap).
  Status ToHost(void* values, uint8_t* validity, int64_t* null_count) const;
  // Arrow C Device Data Interface (include/arrowgpu_cdata.h).  Export shares the buffers: the exported
  // struct keeps them alive until the consumer calls release.  Import takes ownership of `in`
  // (moves it; in->array.release is called when the last buffer reference is dropped) and makes the
  // default stream wait on its sync_event.  Dictionary arrays are not exported (ErrNotImplemented).
  Status ExportDevice(struct ArrowDeviceArray* out, struct ArrowSchema* out_schema) const;
  static Status ImportDevice(struct ArrowDeviceArray* in, const struct ArrowSchema* schema, std::shared_ptr<ArrayData>* out);
};

struct ChunkedArray {  // arrow.Chunked (arrow/table.go:135-143)
  Type type = Type::NA;
  std::vector<std::shared_ptr<ArrayData>> chunks;
  int64_t length = 0;
  int64_t NullN() const;
};

struct Scalar {  // scalar.PrimitiveScalar: Data() is the raw little-endian value
  Type type = Type::NA;
  bool valid = false;
  uint8_t value[8] = {0};
};

namespace compute {

enum class DatumKind { NONE, SCALAR, ARRAY, CHUNKED };  // datum.go KindScalar/KindArray/KindChunked

struct Datum {
  DatumKind kind = DatumKind::NONE;
  std::shared_ptr<Scalar> scalar;
  std::shared_ptr<ArrayData> array;
  std::shared_ptr<ChunkedArray> chunked;
  Datum() = default;
  explicit Datum(std::shared_ptr<ArrayData> a) : kind(DatumKind::ARRAY), array(std::move(a)) {}
  explicit Datum(std::shared_ptr<ChunkedArray> c) : kind(DatumKind::CHUNKED), chunked(std::move(c)) {}
  explicit Datum(std::shared_ptr<Scalar> s) : kind(DatumKind::SCALAR), scalar(std::move(s)) {}
  Type type() const;
  int64_t Len() const;  // -1 for scalars (datum.go: scalars have no length)
};

}  // namespace compute

// ======================================================================================
// exec: the kernel ABI (arrow/compute/exec)
// ======================================================================================
namespace exec {

struct BufferSpan {  // exec/span.go:32-50
  uint8_t* buf = nullptr;  // DEVICE pointer
  int64_t len = 0;         // bytes
  std::shared_ptr<Buffer> owner;
  bool self_alloc = false;
};

struct ArraySpan {  // exec/span.go:76-88
  Type type = Type::NA;
  int64_t len = 0;
  int64_t nulls = 0;
  int64_t offset = 0;
  BufferSpan buffers[2];
  void SetMembers(const ArrayData& d);           // span.go:136-197 (reverse direction of MakeData)
  void SetSlice(int64_t off, int64_t length);    // span.go:208-227
  bool MayHaveNulls() const { return nulls != 0 && buffers[0].buf != nullptr; }  // span.go:105-107
  Status UpdateNullCount(int64_t* out);          // span.go:112-125 (device popcount)
  std::shared_ptr<ArrayData> MakeData() const;   // span.go:136-197
};
using ExecResult = ArraySpan;  // span.go:566

struct ExecValue {  // span.go:548-554
  ArraySpan array;
  const Scalar* scalar = nullptr;
  bool IsArray() const { return scalar == nullptr; }
  bool IsScalar() const { return scalar != nullptr; }
  Type type() const { return scalar ? scalar->type : array.type; }
};

struct ExecSpan {  // span.go:573-576
  int64_t len = 0;
  std::vector<ExecValue> values;
};

enum class NullHandling { INTERSECTION = 0, COMPUTED_PREALLOC = 1, COMPUTED_NO_PREALLOC = 2, OUTPUT_NOT_NULL = 3 };  // kernel.go:457-476
enum class MemAlloc { PREALLOC = 0, NO_PREALLOC = 1 };                                                              // kernel.go:480-499

struct Kernel;
struct KernelCtx {  // kernel.go:40-100
  const Kernel* kernel = nullptr;
  const void* state = nullptr;     // KernelState: the function's options (FilterOptions / TakeOptions ...)
  int64_t* error_word = nullptr;   // device int64, lowered by checked kernels (first failing row); read once per call
  int64_t row_base = 0;            // global row of the span's first row (for error positions)
  Status Allocate(int64_t nbytes, std::shared_ptr<Buffer>* out) const { return Buffer::Allocate(nbytes, out); }
  Status AllocateBitmap(int64_t nbits, std::shared_ptr<Buffer>* out) const { return Buffer::Allocate((nbits + 7) / 8, out); }
};

using ArrayKernelExec = std::function<Status(KernelCtx*, const ExecSpan&, ExecResult*)>;  // kernel.go:617

struct Kernel {
  std::vector<Type> in_types;  // exact-type signature (InputType ExactType matcher); empty entry list = any
  bool any_input_type = false;
  std::function<Type(const std::vector<Type>&)> out_type;  // OutputType resolver (first-arg type, fixed bool, ...)
  ArrayKernelExec exec;
  NullHandling null_handling = NullHandling::INTERSECTION;
  MemAlloc mem_alloc = MemAlloc::PREALLOC;
};
using BatchKernelExec = std::function<Status(KernelCtx*, const std::vector<ExecSpan>&, std::vector<ExecResult>&)>;
struct ScalarKernel : Kernel {  // kernel.go:632-640
  bool can_write_into_slices = true;
  // B200-first extension: when set, the executor hands ALL aligned spans of a chunked call to the
  // kernel at once (one launch, include/arrowgpu.h ag_arith_binary_spans_dev) instead of calling
  // `exec` once per span like executeSpans does (executor.go:598-623).  Same results.
  BatchKernelExec exec_batch;
  bool can_fail = false;        // kernels that lower KernelCtx::error_word
  const char* fail_message = "";
};
struct VectorKernel : Kernel {  // kernel.go:693-704
  bool can_execute_chunkwise = true;
  // ExecChunked (kernel.go:687-691): a non-chunkwise kernel that consumes a whole chunked argument as
  // ONE logical sequence and produces one output array (cumulative_sum, vector_cumulative.go:385-410)
  std::function<Status(KernelCtx*, const ChunkedArray&, ExecResult*)> exec_chunked;
};

}  // namespace exec

// ======================================================================================
// compute: functions, registry, executors (arrow/compute)
// ======================================================================================
namespace compute {

struct FunctionOptions { virtual ~FunctionOptions() = default; virtual const char* TypeName() const = 0; };
struct ArithmeticOptions : FunctionOptions {  // expression.go:480-482
  bool NoCheckOverflow = false;
  const char* TypeName() const override { return "ArithmeticOptions"; }
};
enum NullSelectionBehavior { DropNulls = 0, EmitNulls = 1 };  // kernels/vector_selection.go:34-39
struct FilterOptions : FunctionOptions {
  NullSelectionBehavior NullSelection = DropNulls;
  const char* TypeName() const override { return "FilterOptions"; }
};
struct TakeOptions : FunctionOptions {  // expression.go:494: default BoundsCheck = true
  bool BoundsCheck = true;
  const char* TypeName() const override { return "TakeOptions"; }
};

struct CastOptions : FunctionOptions {  // kernels/cast.go:27-35 (the numeric knobs)
  Type ToType = Type::NA;
  bool AllowIntOverflow = false;
  bool AllowFloatTruncate = false;
  const char* TypeName() const override { return "CastOptions"; }
};
inline CastOptions SafeCastOptions(Type to) { CastOptions o; o.ToType = to; return o; }  // cast.go: SafeCastOptions
inline CastOptions UnsafeCastOptions(Type to) { CastOptions o; o.ToType = to; o.AllowIntOverflow = o.AllowFloatTruncate = true; return o; }

struct CumulativeOptions : FunctionOptions {  // kernels/vector_cumulative.go:92-99
  std::shared_ptr<Scalar> Start;  // nullptr = zero of the input type; a null scalar is invalid
  bool SkipNulls = false;
  const char* TypeName() const override { return "CumulativeOptions"; }
};

enum SortOrder { Ascending = 0, Descending = 1 };            // kernels/vector_sort.go:30-36
enum NullPlacement { NullsAtEnd = 0, NullsAtStart = 1 };     // :38-44
struct SortOptions : FunctionOptions {                        // :46-50 (single key: ColumnIndex is meaningless for an array)
  SortOrder Order = Ascending;
  NullPlacement Placement = NullsAtEnd;
  const char* TypeName() const override { return "SortOptions"; }
};
enum NullMatchingBehavior { NullMatchingMatch = 0, NullMatchingSkip = 1, NullMatchingEmitNull = 2, NullMatchingInconclusive = 3 };
struct Datum;
struct SetLookupOptions : FunctionOptions {                   // compute/scalar_set_lookup.go (ValueSet, NullBehavior)
  std::shared_ptr<ArrayData> ValueSet;
  NullMatchingBehavior NullBehavior = NullMatchingMatch;
  const char* TypeName() const override { return "SetLookupOptions"; }
};

enum NullEncodingBehavior { NullEncodingMask = 0, NullEncodingEncode = 1 };   // kernels/vector_hash.go:83-91
struct DictionaryEncodeOptions : FunctionOptions {                           // :93-98
  NullEncodingBehavior NullEncoding = NullEncodingMask;
  const char* TypeName() const override { return "DictionaryEncodeOptions"; }
};

enum class FuncKind { SCALAR, VECTOR, META };  // functions.go FuncScalar / FuncVector / FuncMeta

class FunctionRegistry;
struct ExecCtx {  // executor.go:46-64
  int64_t ChunkSize = INT64_MAX;
  bool PreallocContiguous = true;
  FunctionRegistry* Registry = nullptr;  // nullptr = GetFunctionRegistry()
};

class Function {  // functions.go:30-41
 public:
  Function(std::string name, FuncKind kind, int arity) : name_(std::move(name)), kind_(kind), arity_(arity) {}
  virtual ~Function() = default;
  const std::string& Name() const { return name_; }
  FuncKind Kind() const { return kind_; }
  int Arity() const { return arity_; }
  virtual Status Execute(const ExecCtx& ctx, const FunctionOptions* opts, const std::vector<Datum>& args, Datum* out) const = 0;
 private:
  std::string name_;
  FuncKind kind_;
  int arity_;
};

class ScalarFunction : public Function {  // functions.go:233-310
 public:
  ScalarFunction(std::string name, int arity) : Function(std::move(name), FuncKind::SCALAR, arity) {}
  Status AddKernel(exec::ScalarKernel k);                                        // functions.go:290
  Status DispatchExact(const std::vector<Type>& types, const exec::ScalarKernel** out) const;  // functions.go:204-217 (first match)
  // arithmeticFunction.DispatchBest (arithmetic.go:112-140) / compareFunction.DispatchBest (scalar_compare.go:37-65):
  // exact match first; binary functions flagged `promote_numeric` then replace both types by
  // commonNumeric (utils.go:178-240).  `types` is rewritten to the dispatched signature.
  Status DispatchBest(std::vector<Type>* types, const exec::ScalarKernel** out) const;
  bool promote_numeric = false;
  Status Execute(const ExecCtx& ctx, const FunctionOptions* opts, const std::vector<Datum>& args, Datum* out) const override;
 private:
  std::vector<exec::ScalarKernel> kernels_;
};

class VectorFunction : public Function {
 public:
  VectorFunction(std::string name, int arity) : Function(std::move(name), FuncKind::VECTOR, arity) {}
  Status AddKernel(exec::VectorKernel k);
  Status DispatchExact(const std::vector<Type>& types, const exec::VectorKernel** out) const;
  Status Execute(const ExecCtx& ctx, const FunctionOptions* opts, const std::vector<Datum>& args, Datum* out) const override;
 private:
  std::vector<exec::VectorKernel> kernels_;
};

class MetaFunction : public Function {  // functions.go:385-430
 public:
  using Impl = std::function<Status(const ExecCtx&, const FunctionOptions*, const std::vector<Datum>&, Datum*)>;
  MetaFunction(std::string name, int arity, Impl impl) : Function(std::move(name), FuncKind::META, arity), impl_(std::move(impl)) {}
  Status Execute(const ExecCtx& ctx, const FunctionOptions* opts, const std::vector<Datum>& args, Datum* out) const override {
    return impl_(ctx, opts, args, out);
  }
 private:
  Impl impl_;
};

class FunctionRegistry {  // registry.go:30-133
 public:
  explicit FunctionRegistry(FunctionRegistry* parent = nullptr) : parent_(parent) {}
  Status AddFunction(std::shared_ptr<Function> fn, bool allow_overwrite);     // registry.go:97
  Status AddAlias(const std::string& target, const std::string& source);     // registry.go:107
  const Function* GetFunction(const std::string& name) const;                // child first, then parent (:120-133)
  std::vector<std::string> GetFunctionNames() const;
 private:
  FunctionRegistry* parent_;
  std::map<std::string, std::shared_ptr<Function>> fns_;
};
FunctionRegistry* GetFunctionRegistry();                                       // registry.go:47-62
std::unique_ptr<FunctionRegistry> NewChildRegistry(FunctionRegistry* parent);  // registry.go:69

// utils.go:178-240; Type::NA when there is no common numeric type
Type CommonNumeric(const std::vector<Type>& types);
// cast.go:919-921: CallFunction("cast") — arrays, chunked arrays and scalars between the 10 numeric types
Status CastDatum(const ExecCtx& ctx, const Datum& val, const CastOptions& opts, Datum* out);

// exec.go:191
Status CallFunction(const ExecCtx& ctx, const std::string& name, const FunctionOptions* opts, const std::vector<Datum>& args, Datum* out);

// arithmetic.go:1090-1142 — default options call the checked function ("add"), NoCheckOverflow the "_unchecked" one
Status Add(const ExecCtx& ctx, const ArithmeticOptions& opts, const Datum& l, const Datum& r, Datum* out);
Status Subtract(const ExecCtx& ctx, const ArithmeticOptions& opts, const Datum& l, const Datum& r, Datum* out);
Status Multiply(const ExecCtx& ctx, const ArithmeticOptions& opts, const Datum& l, const Datum& r, Datum* out);
// vector_cumulative.go:96-102
Status CumulativeSum(const ExecCtx& ctx, const CumulativeOptions& opts, const Datum& values, Datum* out);
Status CumulativeSumChecked(const ExecCtx& ctx, const CumulativeOptions& opts, const Datum& values, Datum* out);
// selection.go:657 / :304
Status Filter(const ExecCtx& ctx, const Datum& values, const Datum& filter, const FilterOptions& opts, Datum* out);
Status Take(const ExecCtx& ctx, const TakeOptions& opts, const Datum& values, const Datum& indices, Datum* out);
// compute.SortIndices (vector_sort.go:205-211), compute.Unique (vector_hash.go), compute.IsIn (scalar_set_lookup.go)
Status SortIndices(const ExecCtx& ctx, const Datum& input, const SortOptions& opts, Datum* out);
Status Unique(const ExecCtx& ctx, const Datum& values, Datum* out);
Status IsIn(const ExecCtx& ctx, const SetLookupOptions& opts, const Datum& values, Datum* out);
// compute.DictionaryEncode (vector_hash.go): a DICTIONARY array (one per chunk of a chunked input, all sharing one
// dictionary) of the 10 numeric types; a dictionary input is returned unchanged
Status DictionaryEncode(const ExecCtx& ctx, const DictionaryEncodeOptions& opts, const Datum& values, Datum* out);

// ---- executor internals exposed for tests (exec_internals_test.go exercises the same pieces) ----
struct SpanPiece { int64_t pos; int64_t len; std::vector<int> chunk_index; std::vector<int64_t> chunk_pos; };
// iterateExecSpans (executor.go:757-863) over per-argument chunk lengths (a one-element vector for a
// plain array, an empty vector for a scalar).
Status IterateExecSpans(const std::vector<std::vector<int64_t>>& arg_chunk_lengths, const std::vector<bool>& is_chunked,
                        int64_t max_chunk_size, std::vector<SpanPiece>* out);
enum class NullGen { PERHAPS_NULL = 0, ALL_VALID = 1, ALL_NULL = 2 };  // executor.go:182-188
NullGen GetNullGen(const exec::ExecValue& v);                         // executor.go:190-214
Status PropagateNulls(exec::KernelCtx* ctx, const exec::ExecSpan& batch, exec::ArraySpan* out);  // executor.go:237-349

}  // namespace compute

// ======================================================================================
// math: arrow/math Sum (validity ignored; operates on values[offset:offset+len])
// ======================================================================================
namespace math {
Status SumFloat64(const ArrayData& a, double* out);    // Float64Funcs.Sum, arrow/math/float64.go:34-39
Status SumInt64(const ArrayData& a, int64_t* out);     // Int64Funcs.Sum
Status SumUint64(const ArrayData& a, uint64_t* out);   // Uint64Funcs.Sum
// Reference-association-order mode: bit-exact with the reference's AVX2 path on any data.
Status SumFloat64ReferenceOrder(const ArrayData& a, double* out);
}  // namespace math

// ======================================================================================
// ipc: Arrow IPC file -> device-resident record batches (arrow/ipc/file_reader.go), and the
// ArrowDeviceArrayStream hand-off of whole batches (arrow/cdata/abi.h:170-200)
// ======================================================================================
namespace ipc {
struct Field { std::string name; Type type = Type::NA; bool nullable = false; };   // arrow.Field of a numeric / boolean column
// Where a column's buffers sit inside its record batch body (offsets relative to the body; -1 = no buffer).
struct ColumnLayout { int64_t length, null_count, validity_offset, validity_length, data_offset, data_length; };
struct RecordBatch { int64_t num_rows = 0; std::vector<std::shared_ptr<ArrayData>> columns; };

class FileReader {
 public:
  ~FileReader();
  // NewMappedFileReader (file_reader.go:231-250): `data` (a memory map or a pinned slab) must outlive the reader.
  static Status Open(const uint8_t* data, int64_t size, std::unique_ptr<FileReader>* out);
  const std::vector<Field>& schema() const;   // FileReader.Schema :383
  int NumRecords() const;                     // :394
  int version() const;                        // MetadataVersion :398
  // Metadata of record batch i only — no device work: the checks of validateFileBlock :68-99,
  // validateFileBlockMetadata (metadata.go:78-109) and newRecordBatch's buffer walk :523-575, 732-780.
  Status Layout(int i, int64_t* num_rows, int64_t* body_offset, int64_t* body_length, std::vector<ColumnLayout>* cols) const;
  // RecordBatchAt :451-480.  The batch body crosses the link ONCE (one H2D copy); columns are views into it.
  Status RecordBatchAt(int i, RecordBatch* out) const;
 private:
  FileReader();
  struct Impl;
  Impl* impl_;
};

// Producer: every get_next reads the next record batch of `reader` (one H2D copy) and hands it over as a struct-typed
// ArrowDeviceArray {ARROW_DEVICE_CUDA, current device} whose children are the columns.  The stream owns the reader.
Status ExportDeviceStream(std::shared_ptr<FileReader> reader, struct ArrowDeviceArrayStream* out);
// Consumer: drains a device stream (ours or another producer's) into record batches; columns keep the producer's
// arrays alive until the last reference goes (release is called then).  Calls stream->release at the end.
Status ImportDeviceStream(struct ArrowDeviceArrayStream* stream, std::vector<Field>* schema, std::vector<RecordBatch>* out);
}  // namespace ipc

}  // namespace arrowgpu
