// compute.cc — host-side mirror of arrow-go's compute executors and function registry driving
// the device kernels of libarrowgpu.so.  See arrowgpu_compute.h for the reference map.
#include "arrowgpu_compute.h"

#include <string.h>
#include <algorithm>
#include <mutex>

namespace arrowgpu {

// ---------------------------------------------------------------- types -------------------
int BitWidth(Type t) {
  switch (t) {
    case Type::BOOL: return 1;
    case Type::UINT8: case Type::INT8: return 8;
    case Type::UINT16: case Type::INT16: case Type::FLOAT16: return 16;
    case Type::UINT32: case Type::INT32: case Type::FLOAT32: return 32;
    case Type::UINT64: case Type::INT64: case Type::FLOAT64: return 64;
    default: return 0;  // DICTIONARY included: its int32 indices are not values of the array's type
  }
}
const char* TypeName(Type t) {
  static const char* names[] = {"null", "bool", "uint8", "int8", "uint16", "int16", "uint32", "int32", "uint64", "int64", "float16", "float32", "float64"};
  const int i = (int)t;
  if (t == Type::DICTIONARY) return "dictionary";
  return (i >= 0 && i <= 12) ? names[i] : "unknown";
}
bool IsSignedInteger(Type t) { return t == Type::INT8 || t == Type::INT16 || t == Type::INT32 || t == Type::INT64; }
bool IsInteger(Type t) { return IsSignedInteger(t) || t == Type::UINT8 || t == Type::UINT16 || t == Type::UINT32 || t == Type::UINT64; }
bool IsFloating(Type t) { return t == Type::FLOAT32 || t == Type::FLOAT64; }
bool IsNumeric(Type t) { return IsInteger(t) || IsFloating(t); }

Status Status::FromNative(int c) {
  if (c == AG_OK) return OK();
  char buf[512];
  ag_last_error(buf, sizeof(buf));
  return Make(c, buf);
}

#define RETURN_NOT_OK(expr)                \
  do {                                     \
    ::arrowgpu::Status _st = (expr);       \
    if (!_st.ok()) return _st;             \
  } while (0)
#define NATIVE(expr)                                            \
  do {                                                          \
    int _c = (expr);                                            \
    if (_c != AG_OK) return ::arrowgpu::Status::FromNative(_c); \
  } while (0)

static inline int64_t BytesForBits(int64_t n) { return (n + 7) / 8; }
static inline int64_t DataBytes(Type t, int64_t n) { return t == Type::BOOL ? BytesForBits(n) : n * (BitWidth(t) / 8); }

// ---------------------------------------------------------------- Buffer ------------------
Buffer::~Buffer() {
  if (foreign_) { if (on_release_) on_release_(); }
  else if (data_) ag_dev_free(data_);
}

std::shared_ptr<Buffer> Buffer::Wrap(const void* device_ptr, int64_t nbytes, std::function<void()> on_release) {
  auto b = std::shared_ptr<Buffer>(new Buffer());
  b->data_ = const_cast<uint8_t*>(static_cast<const uint8_t*>(device_ptr));
  b->size_ = nbytes;
  b->foreign_ = true;
  b->on_release_ = std::move(on_release);
  return b;
}

Status Buffer::Allocate(int64_t nbytes, std::shared_ptr<Buffer>* out) {
  auto b = std::shared_ptr<Buffer>(new Buffer());
  void* p = nullptr;
  NATIVE(ag_dev_alloc(&p, (size_t)(nbytes + 8)));  // +8: bitmap kernels address whole 32-bit words
  b->data_ = (uint8_t*)p;
  b->size_ = nbytes;
  *out = std::move(b);
  return Status::OK();
}
Status Buffer::FromHost(const void* host, int64_t nbytes, std::shared_ptr<Buffer>* out) {
  RETURN_NOT_OK(Allocate(nbytes, out));
  if (nbytes) {
    NATIVE(ag_upload((*out)->data(), host, (size_t)nbytes, nullptr));
    NATIVE(ag_stream_sync(nullptr));
  }
  return Status::OK();
}
Status Buffer::ToHost(void* host, int64_t nbytes, int64_t byte_offset) const {
  if (nbytes) {
    NATIVE(ag_download(host, data_ + byte_offset, (size_t)nbytes, nullptr));
    NATIVE(ag_stream_sync(nullptr));
  }
  return Status::OK();
}

// ---------------------------------------------------------------- ArrayData ---------------
namespace {
struct ExportedBuffers { std::shared_ptr<Buffer> b[2]; };
void ReleaseExportedBuffers(void* opaque) { delete static_cast<ExportedBuffers*>(opaque); }
}  // namespace

Status ArrayData::ExportDevice(struct ArrowDeviceArray* out, struct ArrowSchema* out_schema) const {
  if (type == Type::DICTIONARY) return Status::NotImplemented("export: dictionary arrays are not exported through the C Device Data Interface");
  auto* keep = new ExportedBuffers{{buffers[0], buffers[1]}};
  const int rc = ag_export_device_array((int)type, length, null_count, offset, buffers[0] ? buffers[0]->data() : nullptr,
                                        buffers[1] ? buffers[1]->data() : nullptr, ReleaseExportedBuffers, keep, nullptr, out, out_schema);
  if (rc != AG_OK) { delete keep; return Status::FromNative(rc); }
  return Status::OK();
}

Status ArrayData::ImportDevice(struct ArrowDeviceArray* in, const struct ArrowSchema* schema, std::shared_ptr<ArrayData>* out) {
  ag_array_view v;
  NATIVE(ag_import_device_array(in, schema, nullptr, &v));
  if (v.type == 0) return Status::Invalid("import: a schema is required");
  // move the struct: the importer owns it now (C Data Interface "moving an array")
  auto owned = std::make_shared<ArrowDeviceArray>(*in);
  in->array.release = nullptr;
  auto releaser = std::shared_ptr<void>(nullptr, [owned](void*) { if (owned->array.release) owned->array.release(&owned->array); });
  auto d = std::make_shared<ArrayData>();
  d->type = (Type)v.type; d->length = v.length; d->offset = v.offset; d->null_count = v.null_count;
  const int64_t n = v.offset + v.length;
  if (v.validity) d->buffers[0] = Buffer::Wrap(v.validity, BytesForBits(n), [releaser] {});
  d->buffers[1] = Buffer::Wrap(v.values, DataBytes((Type)v.type, n), [releaser] {});
  if (!v.validity) d->null_count = 0;
  *out = d;
  return Status::OK();
}

std::shared_ptr<ArrayData> ArrayData::Slice(int64_t off, int64_t len) const {
  auto d = std::make_shared<ArrayData>(*this);
  d->offset = offset + off;
  d->length = len;
  // array.NewSliceData: a slice of an array with nulls has an unknown null count
  if (null_count != 0 && !(off == 0 && len == length)) d->null_count = (null_count == length) ? len : kUnknownNullCount;
  return d;
}

Status ArrayData::FromHost(Type type, int64_t length, int64_t offset, const uint8_t* validity, const void* values,
                           int64_t null_count, std::shared_ptr<ArrayData>* out) {
  if (BitWidth(type) == 0) return Status::TypeError(std::string("unsupported type ") + TypeName(type));
  if (length < 0 || offset < 0) return Status::Invalid("negative length or offset");
  auto d = std::make_shared<ArrayData>();
  d->type = type; d->length = length; d->offset = offset; d->null_count = validity ? null_count : 0;
  RETURN_NOT_OK(Buffer::FromHost(values, DataBytes(type, offset + length), &d->buffers[1]));
  if (validity) RETURN_NOT_OK(Buffer::FromHost(validity, BytesForBits(offset + length), &d->buffers[0]));
  *out = std::move(d);
  return Status::OK();
}

Status ArrayData::ToHost(void* values, uint8_t* validity, int64_t* null_count_out) const {
  if (length == 0) { if (null_count_out) *null_count_out = 0; return Status::OK(); }
  const int w = type == Type::DICTIONARY ? 32 : BitWidth(type);
  if (values) {
    if (type == Type::BOOL) {
      // re-base to bit 0 on the device, then copy
      std::shared_ptr<Buffer> tmp;
      RETURN_NOT_OK(Buffer::Allocate(BytesForBits(length), &tmp));
      NATIVE(ag_bitmap_copy_dev(buffers[1]->data(), offset, length, tmp->data(), 0, nullptr));
      RETURN_NOT_OK(tmp->ToHost(values, BytesForBits(length)));
    } else {
      RETURN_NOT_OK(buffers[1]->ToHost(values, length * (w / 8), offset * (w / 8)));
    }
  }
  int64_t nulls = null_count;
  if (buffers[0]) {
    std::shared_ptr<Buffer> tmp;
    RETURN_NOT_OK(Buffer::Allocate(BytesForBits(length) + 8, &tmp));
    NATIVE(ag_bitmap_copy_dev(buffers[0]->data(), offset, length, tmp->data(), 0, nullptr));
    if (validity) RETURN_NOT_OK(tmp->ToHost(validity, BytesForBits(length)));
    if (nulls == kUnknownNullCount) {
      int64_t* cnt = (int64_t*)(tmp->data() + ((BytesForBits(length) + 7) & ~7ll));
      std::shared_ptr<Buffer> cbuf;
      RETURN_NOT_OK(Buffer::Allocate(8, &cbuf));
      (void)cnt;
      NATIVE(ag_bitmap_popcount_dev(buffers[0]->data(), offset, length, (int64_t*)cbuf->data(), nullptr));
      int64_t set = 0;
      RETURN_NOT_OK(cbuf->ToHost(&set, 8));
      nulls = length - set;
    }
  } else {
    if (validity) memset(validity, 0xff, (size_t)BytesForBits(length));
    nulls = 0;
  }
  if (null_count_out) *null_count_out = nulls;
  return Status::OK();
}

int64_t ChunkedArray::NullN() const {
  int64_t n = 0;
  for (auto& c : chunks) n += (c->null_count == kUnknownNullCount) ? 1 : c->null_count;  // "may have nulls"
  return n;
}

namespace compute {
Type Datum::type() const {
  switch (kind) {
    case DatumKind::SCALAR: return scalar->type;
    case DatumKind::ARRAY: return array->type;
    case DatumKind::CHUNKED: return chunked->type;
    default: return Type::NA;
  }
}
int64_t Datum::Len() const {
  switch (kind) {
    case DatumKind::ARRAY: return array->length;
    case DatumKind::CHUNKED: return chunked->length;
    default: return -1;
  }
}
}  // namespace compute

// ======================================================================================
// exec::ArraySpan
// ======================================================================================
namespace exec {

void ArraySpan::SetMembers(const ArrayData& d) {
  type = d.type; len = d.length; nulls = d.null_count; offset = d.offset;
  for (int i = 0; i < 2; ++i) {
    buffers[i] = BufferSpan();
    if (d.buffers[i]) {
      buffers[i].buf = d.buffers[i]->data();
      buffers[i].len = d.buffers[i]->size();
      buffers[i].owner = d.buffers[i];
    }
  }
  if (!buffers[0].buf && type != Type::NA) nulls = 0;  // no validity bitmap => no nulls
}

void ArraySpan::SetSlice(int64_t off, int64_t length) {
  if (off == offset && length == len) return;
  if (type != Type::NA) {
    if (nulls != 0) nulls = (nulls == len) ? length : kUnknownNullCount;
  } else {
    nulls = length;
  }
  offset = off; len = length;
}

Status ArraySpan::UpdateNullCount(int64_t* out) {
  if (nulls != kUnknownNullCount) { if (out) *out = nulls; return Status::OK(); }
  if (!buffers[0].buf || buffers[0].len == 0) { nulls = 0; if (out) *out = 0; return Status::OK(); }
  std::shared_ptr<Buffer> cnt;
  RETURN_NOT_OK(Buffer::Allocate(8, &cnt));
  NATIVE(ag_bitmap_popcount_dev(buffers[0].buf, offset, len, (int64_t*)cnt->data(), nullptr));
  int64_t set = 0;
  RETURN_NOT_OK(cnt->ToHost(&set, 8));
  nulls = len - set;
  if (out) *out = nulls;
  return Status::OK();
}

std::shared_ptr<ArrayData> ArraySpan::MakeData() const {
  auto d = std::make_shared<ArrayData>();
  d->type = type; d->length = len; d->null_count = nulls; d->offset = offset;
  for (int i = 0; i < 2; ++i) d->buffers[i] = buffers[i].owner;
  if (!d->buffers[0]) d->null_count = 0;
  return d;
}

}  // namespace exec

// ======================================================================================
// compute: null propagation, span iteration, executors
// ======================================================================================
namespace compute {

using exec::ArraySpan;
using exec::ExecSpan;
using exec::ExecValue;
using exec::KernelCtx;

NullGen GetNullGen(const ExecValue& v) {  // executor.go:190-214
  if (v.type() == Type::NA) return NullGen::ALL_NULL;
  if (v.IsScalar()) return v.scalar->valid ? NullGen::ALL_VALID : NullGen::ALL_NULL;
  const ArraySpan& arr = v.array;
  // do not count if they haven't been counted already
  if (arr.nulls == 0 || arr.buffers[0].buf == nullptr) return NullGen::ALL_VALID;
  if (arr.nulls == arr.len) return NullGen::ALL_NULL;
  return NullGen::PERHAPS_NULL;
}

static NullGen GetNullGenDatum(const Datum& d) {  // executor.go:216-230
  if (d.kind == DatumKind::CHUNKED) return NullGen::PERHAPS_NULL;
  ExecValue v;
  if (d.kind == DatumKind::ARRAY) v.array.SetMembers(*d.array);
  else v.scalar = d.scalar.get();
  return GetNullGen(v);
}

Status PropagateNulls(KernelCtx* ctx, const ExecSpan& batch, ArraySpan* out) {  // executor.go:237-349
  if (out->type == Type::NA) return Status::OK();
  if (out->offset != 0 && out->buffers[0].buf == nullptr)
    return Status::Invalid("can only propagate nulls into pre-allocated memory when output offset is non-zero");
  std::vector<const ArraySpan*> arrs_with_nulls;
  bool is_all_null = false;
  const bool prealloc = out->buffers[0].buf != nullptr;
  for (auto& v : batch.values) {
    const NullGen g = GetNullGen(v);
    if (g == NullGen::ALL_NULL) is_all_null = true;
    if (g != NullGen::ALL_VALID && v.IsArray()) arrs_with_nulls.push_back(&v.array);
  }
  auto alloc_bitmap = [&]() -> Status {
    std::shared_ptr<Buffer> buf;
    RETURN_NOT_OK(ctx->AllocateBitmap(out->len + out->offset, &buf));
    out->buffers[0].buf = buf->data(); out->buffers[0].len = buf->size(); out->buffers[0].owner = buf; out->buffers[0].self_alloc = true;
    return Status::OK();
  };
  if (is_all_null) {
    out->nulls = out->len;
    if (prealloc) { NATIVE(ag_bitmap_set_dev(out->buffers[0].buf, out->offset, out->len, 0, nullptr)); return Status::OK(); }
    for (auto* arr : arrs_with_nulls) {
      if (arr->nulls == arr->len && arr->buffers[0].owner) { out->buffers[0] = arr->buffers[0]; return Status::OK(); }
    }
    RETURN_NOT_OK(alloc_bitmap());
    NATIVE(ag_bitmap_set_dev(out->buffers[0].buf, out->offset, out->len, 0, nullptr));
    return Status::OK();
  }
  out->nulls = kUnknownNullCount;
  switch (arrs_with_nulls.size()) {
    case 0:
      out->nulls = 0;
      if (prealloc) NATIVE(ag_bitmap_set_dev(out->buffers[0].buf, out->offset, out->len, 1, nullptr));
      return Status::OK();
    case 1: {
      const ArraySpan* arr = arrs_with_nulls[0];
      out->nulls = arr->nulls;
      if (prealloc) {
        NATIVE(ag_bitmap_copy_dev(arr->buffers[0].buf, arr->offset, arr->len, out->buffers[0].buf, out->offset, nullptr));
        return Status::OK();
      }
      if (arr->offset == 0) { out->buffers[0] = arr->buffers[0]; out->buffers[0].self_alloc = false; return Status::OK(); }  // zero-copy share
      // (the reference also zero-copies byte-aligned offsets with SliceBuffer; a device Buffer has no
      //  sub-buffer view here, so those are copied like the unaligned case — same bits)
      RETURN_NOT_OK(alloc_bitmap());
      NATIVE(ag_bitmap_copy_dev(arr->buffers[0].buf, arr->offset, arr->len, out->buffers[0].buf, 0, nullptr));
      return Status::OK();
    }
    default: {
      if (!prealloc) RETURN_NOT_OK(alloc_bitmap());
      uint8_t* ob = out->buffers[0].buf;
      NATIVE(ag_bitmap_op_dev(AG_BITOP_AND, arrs_with_nulls[0]->buffers[0].buf, arrs_with_nulls[0]->offset,
                              arrs_with_nulls[1]->buffers[0].buf, arrs_with_nulls[1]->offset, ob, out->offset, out->len, nullptr));
      for (size_t i = 2; i < arrs_with_nulls.size(); ++i)
        NATIVE(ag_bitmap_op_dev(AG_BITOP_AND, ob, out->offset, arrs_with_nulls[i]->buffers[0].buf, arrs_with_nulls[i]->offset,
                                ob, out->offset, out->len, nullptr));
      return Status::OK();
    }
  }
}

// iterateExecSpans, executor.go:757-863, on chunk lengths only (metadata): testable without a GPU.
Status IterateExecSpans(const std::vector<std::vector<int64_t>>& lens, const std::vector<bool>& is_chunked,
                        int64_t max_chunk_size, std::vector<SpanPiece>* out) {
  out->clear();
  const size_t nargs = lens.size();
  int64_t length = -1;
  bool all_same = true;
  for (size_t i = 0; i < nargs; ++i) {
    if (lens[i].empty() && !is_chunked[i]) continue;  // scalar
    int64_t tot = 0;
    for (int64_t l : lens[i]) tot += l;
    if (length < 0) length = tot; else if (length != tot) all_same = false;
  }
  if (length < 0) length = 1;  // all scalars: a single row (checkIfAllScalar / PromoteExecSpanScalars)
  if (!all_same) return Status::Invalid("array args must all be the same length");
  max_chunk_size = std::min(length, max_chunk_size);
  std::vector<int> chunk_idx(nargs, 0);
  std::vector<int64_t> value_pos(nargs, 0);
  int64_t pos = 0;
  while (pos != length) {
    int64_t iter = std::min(length - pos, max_chunk_size);
    for (size_t i = 0; i < nargs && iter > 0; ++i) {
      if (!is_chunked[i]) continue;
      if (lens[i].empty()) { iter = 0; continue; }
      while (value_pos[i] == lens[i][chunk_idx[i]]) { chunk_idx[i]++; value_pos[i] = 0; }  // exhausted or zero-length chunk
      iter = std::min(lens[i][chunk_idx[i]] - value_pos[i], iter);
    }
    SpanPiece p;
    p.pos = pos; p.len = iter; p.chunk_index = chunk_idx; p.chunk_pos = value_pos;
    out->push_back(p);
    for (size_t i = 0; i < nargs; ++i)
      if (!(lens[i].empty() && !is_chunked[i])) value_pos[i] += iter;
    pos += iter;
    if (iter == 0) break;  // degenerate (empty chunked argument)
  }
  return Status::OK();
}

// ---------------------------------------------------------------- registry ----------------
Status FunctionRegistry::AddFunction(std::shared_ptr<Function> fn, bool allow_overwrite) {
  if (!allow_overwrite && fns_.count(fn->Name())) return Status::Make(AG_ERR_INVALID, "already have a function registered with name: " + fn->Name());
  fns_[fn->Name()] = std::move(fn);
  return Status::OK();
}
Status FunctionRegistry::AddAlias(const std::string& target, const std::string& source) {
  const Function* f = GetFunction(source);
  if (!f) return Status::Make(AG_ERR_INVALID, "no function registered with name: " + source);  // arrow.ErrKey
  for (auto& kv : fns_) if (kv.second.get() == f) { fns_[target] = kv.second; return Status::OK(); }
  return Status::Invalid("alias source lives in a parent registry");
}
const Function* FunctionRegistry::GetFunction(const std::string& name) const {
  auto it = fns_.find(name);
  if (it != fns_.end()) return it->second.get();
  return parent_ ? parent_->GetFunction(name) : nullptr;
}
std::vector<std::string> FunctionRegistry::GetFunctionNames() const {
  std::vector<std::string> names = parent_ ? parent_->GetFunctionNames() : std::vector<std::string>();
  for (auto& kv : fns_) names.push_back(kv.first);
  std::sort(names.begin(), names.end());
  names.erase(std::unique(names.begin(), names.end()), names.end());
  return names;
}
std::unique_ptr<FunctionRegistry> NewChildRegistry(FunctionRegistry* parent) { return std::unique_ptr<FunctionRegistry>(new FunctionRegistry(parent)); }

template <typename K>
static Status DispatchFirstMatch(const std::string& fname, const std::vector<K>& kernels, const std::vector<Type>& types, const K** out) {
  for (auto& k : kernels) {  // first match wins (functions.go:209-213)
    if (k.any_input_type) { *out = &k; return Status::OK(); }
    if (k.in_types.size() != types.size()) continue;
    bool ok = true;
    for (size_t i = 0; i < types.size(); ++i) ok = ok && (k.in_types[i] == types[i]);
    if (ok) { *out = &k; return Status::OK(); }
  }
  std::string sig;
  for (size_t i = 0; i < types.size(); ++i) sig += std::string(i ? ", " : "") + TypeName(types[i]);
  return Status::NotImplemented("function '" + fname + "' has no kernel matching input types (" + sig + ")");
}
Status ScalarFunction::AddKernel(exec::ScalarKernel k) {
  if (!k.any_input_type && (int)k.in_types.size() != Arity()) return Status::Invalid("kernel arity does not match function arity");
  kernels_.push_back(std::move(k));
  return Status::OK();
}
Status ScalarFunction::DispatchExact(const std::vector<Type>& types, const exec::ScalarKernel** out) const {
  return DispatchFirstMatch(Name(), kernels_, types, out);
}
// commonNumeric, utils.go:178-240
Type CommonNumeric(const std::vector<Type>& types) {
  for (Type t : types) if (!IsInteger(t) && !IsFloating(t)) return Type::NA;
  for (Type t : types) if (t == Type::FLOAT64) return Type::FLOAT64;
  for (Type t : types) if (t == Type::FLOAT32) return Type::FLOAT32;
  int max_signed = 0, max_unsigned = 0;
  for (Type t : types) {
    if (IsSignedInteger(t)) max_signed = std::max(max_signed, BitWidth(t));
    else max_unsigned = std::max(max_unsigned, BitWidth(t));
  }
  if (max_signed == 0) {
    if (max_unsigned >= 64) return Type::UINT64;
    if (max_unsigned == 32) return Type::UINT32;
    if (max_unsigned == 16) return Type::UINT16;
    return Type::UINT8;
  }
  if (max_signed <= max_unsigned) {  // bitutil.NextPowerOf2(maxWidthUnsigned + 1)
    int w = 1;
    while (w < max_unsigned + 1) w <<= 1;
    max_signed = w;
  }
  if (max_signed >= 64) return Type::INT64;
  if (max_signed == 32) return Type::INT32;
  if (max_signed == 16) return Type::INT16;
  return Type::INT8;
}

Status ScalarFunction::DispatchBest(std::vector<Type>* types, const exec::ScalarKernel** out) const {
  if (DispatchExact(*types, out).ok()) return Status::OK();
  if (promote_numeric && types->size() == 2) {  // "only promote types for binary funcs", arithmetic.go:127-137
    const Type common = CommonNumeric(*types);
    if (common != Type::NA) { (*types)[0] = common; (*types)[1] = common; }
  }
  return DispatchExact(*types, out);
}

Status VectorFunction::AddKernel(exec::VectorKernel k) { kernels_.push_back(std::move(k)); return Status::OK(); }
Status VectorFunction::DispatchExact(const std::vector<Type>& types, const exec::VectorKernel** out) const {
  return DispatchFirstMatch(Name(), kernels_, types, out);
}

// ---------------------------------------------------------------- scalar executor ---------
// A DICTIONARY array is its int32 indices plus a dictionary: no kernel of this layer decodes it, and none may read the
// indices as values of the array's type.
static Status RejectDictionaries(const std::string& fn, const std::vector<Datum>& args) {
  for (auto& a : args)
    if (a.kind != DatumKind::NONE && a.kind != DatumKind::SCALAR && a.type() == Type::DICTIONARY)
      return Status::NotImplemented("function '" + fn + "' does not take dictionary arrays");
  return Status::OK();
}
static Status CheckArgs(const Function& fn, const std::vector<Datum>& args) {
  if ((int)args.size() != fn.Arity())
    return Status::Invalid("function '" + fn.Name() + "' accepts " + std::to_string(fn.Arity()) + " arguments but " + std::to_string(args.size()) + " passed");
  for (auto& a : args) if (a.kind == DatumKind::NONE) return Status::Invalid("tried executing function with non-value type");  // checkAllIsValue
  return RejectDictionaries(fn.Name(), args);
}

namespace {
struct ErrorWord {  // device int64 "first failing row", reset per call
  std::shared_ptr<Buffer> buf;
  Status Init() { RETURN_NOT_OK(Buffer::Allocate(8, &buf)); NATIVE(ag_error_word_reset_dev((int64_t*)buf->data(), nullptr)); return Status::OK(); }
  Status Read(int64_t* v) { return buf->ToHost(v, 8); }
};
}  // namespace

// scalarExecutor: executor.go:487-728 (Init :435-440, setupPrealloc :658-702, executeSpans :598-623,
// executeSingleSpan :644-656, emitResult :704-728) + WrapResults :521-580.
Status ScalarFunction::Execute(const ExecCtx& ectx, const FunctionOptions* opts, const std::vector<Datum>& args_in, Datum* out) const {
  RETURN_NOT_OK(CheckArgs(*this, args_in));
  std::vector<Type> in_types;
  for (auto& a : args_in) in_types.push_back(a.type());
  const exec::ScalarKernel* kernel = nullptr;
  RETURN_NOT_OK(DispatchBest(&in_types, &kernel));
  // "cast arguments if necessary" (exec.go:101-121): implicit promotion runs the safe cast
  std::vector<Datum> cast_args;
  for (size_t i = 0; i < args_in.size(); ++i) {
    if (args_in[i].type() == in_types[i]) continue;
    if (cast_args.empty()) cast_args = args_in;
    RETURN_NOT_OK(CastDatum(ectx, args_in[i], SafeCastOptions(in_types[i]), &cast_args[i]));
  }
  const std::vector<Datum>& args = cast_args.empty() ? args_in : cast_args;
  const Type out_type = kernel->out_type(in_types);

  // span iteration metadata
  std::vector<std::vector<int64_t>> lens(args.size());
  std::vector<bool> is_chunked(args.size(), false);
  bool have_chunked = false, all_scalar = true;
  for (size_t i = 0; i < args.size(); ++i) {
    if (args[i].kind == DatumKind::ARRAY) { lens[i] = {args[i].array->length}; all_scalar = false; }
    else if (args[i].kind == DatumKind::CHUNKED) {
      is_chunked[i] = true; have_chunked = true; all_scalar = false;
      for (auto& c : args[i].chunked->chunks) lens[i].push_back(c->length);
    }
  }
  if (all_scalar) return Status::NotImplemented("scalar-only execution (PromoteExecSpanScalars) is not part of the accelerated path");
  std::vector<SpanPiece> pieces;
  RETURN_NOT_OK(IterateExecSpans(lens, is_chunked, ectx.ChunkSize, &pieces));
  int64_t total = 0;
  for (size_t i = 0; i < args.size(); ++i) if (args[i].kind != DatumKind::SCALAR) { total = args[i].Len(); break; }

  // setupPrealloc (executor.go:658-702)
  bool validity_prealloc = false, elide_validity = false;
  if (out_type != Type::NA) {
    if (kernel->null_handling == exec::NullHandling::COMPUTED_PREALLOC) validity_prealloc = true;
    else if (kernel->null_handling == exec::NullHandling::INTERSECTION) {
      elide_validity = true;
      for (auto& a : args) if (GetNullGenDatum(a) != NullGen::ALL_VALID) { elide_validity = false; break; }
      validity_prealloc = !elide_validity;
    }
  }
  const bool data_prealloc = kernel->mem_alloc == exec::MemAlloc::PREALLOC;
  const bool contiguous = ectx.PreallocContiguous && kernel->can_write_into_slices && data_prealloc &&
                          (validity_prealloc || elide_validity || kernel->null_handling == exec::NullHandling::OUTPUT_NOT_NULL);

  KernelCtx kctx;
  kctx.kernel = kernel;
  kctx.state = opts;
  ErrorWord err_word;
  if (kernel->can_fail) { RETURN_NOT_OK(err_word.Init()); kctx.error_word = (int64_t*)err_word.buf->data(); }

  auto prepare_output = [&](int64_t length, ArraySpan* o) -> Status {  // prepareOutput, executor.go:441-470
    *o = ArraySpan();
    o->type = out_type; o->len = length; o->offset = 0; o->nulls = kUnknownNullCount;
    if (validity_prealloc) {
      std::shared_ptr<Buffer> b;
      RETURN_NOT_OK(kctx.AllocateBitmap(length, &b));
      o->buffers[0].buf = b->data(); o->buffers[0].len = b->size(); o->buffers[0].owner = b; o->buffers[0].self_alloc = true;
    }
    if (data_prealloc) {
      std::shared_ptr<Buffer> b;
      RETURN_NOT_OK(kctx.Allocate(DataBytes(out_type, length), &b));  // allocateDataBuffer, executor.go:155-163
      o->buffers[1].buf = b->data(); o->buffers[1].len = b->size(); o->buffers[1].owner = b; o->buffers[1].self_alloc = true;
    }
    if (kernel->null_handling == exec::NullHandling::OUTPUT_NOT_NULL || elide_validity) o->nulls = 0;
    return Status::OK();
  };

  auto build_span = [&](const SpanPiece& p, ExecSpan* span) {
    span->len = p.len;
    span->values.assign(args.size(), ExecValue());
    for (size_t i = 0; i < args.size(); ++i) {
      ExecValue& v = span->values[i];
      if (args[i].kind == DatumKind::SCALAR) { v.scalar = args[i].scalar.get(); continue; }
      const ArrayData& d = (args[i].kind == DatumKind::ARRAY) ? *args[i].array : *args[i].chunked->chunks[p.chunk_index[i]];
      v.array.SetMembers(d);
      v.array.SetSlice(d.offset + p.chunk_pos[i], p.len);
    }
  };

  auto exec_single = [&](const ExecSpan& span, ArraySpan* o) -> Status {  // executeSingleSpan, executor.go:644-656
    if (o->type != Type::NA && kernel->null_handling == exec::NullHandling::INTERSECTION && !elide_validity)
      RETURN_NOT_OK(PropagateNulls(&kctx, span, o));
    return kernel->exec(&kctx, span, o);
  };

  std::vector<std::shared_ptr<ArrayData>> results;
  if (contiguous) {
    ArraySpan output;
    RETURN_NOT_OK(prepare_output(total, &output));
    const bool batched = static_cast<bool>(kernel->exec_batch) && pieces.size() > 1;
    std::vector<ExecSpan> all_spans;
    std::vector<ArraySpan> all_outs;
    for (auto& p : pieces) {
      if (p.len == 0) continue;
      ExecSpan span;
      build_span(p, &span);
      ArraySpan slice = output;
      slice.SetSlice(p.pos, p.len);       // out.SetSlice(resultOffset, input.Len), executor.go:609
      slice.nulls = kUnknownNullCount;
      kctx.row_base = p.pos;
      if (batched) {
        // validity still goes span by span (bitmap launches are tiny); the value kernel runs once
        if (out_type != Type::NA && kernel->null_handling == exec::NullHandling::INTERSECTION && !elide_validity)
          RETURN_NOT_OK(PropagateNulls(&kctx, span, &slice));
        all_spans.push_back(std::move(span));
        all_outs.push_back(slice);
      } else {
        RETURN_NOT_OK(exec_single(span, &slice));
      }
    }
    if (batched && !all_spans.empty()) RETURN_NOT_OK(kernel->exec_batch(&kctx, all_spans, all_outs));
    output.nulls = (elide_validity || kernel->null_handling == exec::NullHandling::OUTPUT_NOT_NULL) ? 0 : kUnknownNullCount;
    results.push_back(output.MakeData());
  } else {
    for (auto& p : pieces) {
      if (p.len == 0 && pieces.size() > 1) continue;
      ExecSpan span;
      build_span(p, &span);
      ArraySpan o;
      RETURN_NOT_OK(prepare_output(p.len, &o));
      kctx.row_base = p.pos;
      RETURN_NOT_OK(exec_single(span, &o));
      results.push_back(o.MakeData());
    }
  }
  if (results.empty()) {  // zero-length input: one empty output
    ArraySpan o;
    RETURN_NOT_OK(prepare_output(0, &o));
    o.nulls = 0;
    results.push_back(o.MakeData());
  }
  if (kernel->can_fail) {
    int64_t bad = 0;
    RETURN_NOT_OK(err_word.Read(&bad));
    if (bad != AG_NO_ERROR_POS) return Status::Invalid(kernel->fail_message);  // the output is released, exec.go:161-170
  }
  // emitResult :704-708 recounts nulls lazily; we leave them unknown (ToHost counts on demand)
  if (have_chunked) {  // WrapResults: Chunked if any input was chunked (executor.go:521-580)
    auto c = std::make_shared<ChunkedArray>();
    c->type = out_type; c->chunks = results;
    for (auto& r : results) c->length += r->length;
    *out = Datum(c);
  } else {
    *out = Datum(results.empty() ? std::make_shared<ArrayData>() : results[0]);
  }
  return Status::OK();
}

// ---------------------------------------------------------------- vector executor ---------
// vectorExecutor, executor.go:886-1154: chunk-wise kernels run once per aligned span and emit one
// output array per span; non-chunkwise kernels (array_take) need whole arrays.
Status VectorFunction::Execute(const ExecCtx& ectx, const FunctionOptions* opts, const std::vector<Datum>& args, Datum* out) const {
  (void)ectx;
  RETURN_NOT_OK(CheckArgs(*this, args));
  std::vector<Type> in_types;
  for (auto& a : args) in_types.push_back(a.type());
  const exec::VectorKernel* kernel = nullptr;
  RETURN_NOT_OK(DispatchExact(in_types, &kernel));
  const Type out_type = kernel->out_type(in_types);
  KernelCtx kctx;
  kctx.kernel = kernel;
  kctx.state = opts;
  bool have_chunked = false;
  std::vector<std::vector<int64_t>> lens(args.size());
  std::vector<bool> is_chunked(args.size(), false);
  for (size_t i = 0; i < args.size(); ++i) {
    if (args[i].kind == DatumKind::SCALAR) return Status::NotImplemented("vector kernels take array-like arguments");
    if (args[i].kind == DatumKind::ARRAY) lens[i] = {args[i].array->length};
    else { is_chunked[i] = true; have_chunked = true; for (auto& c : args[i].chunked->chunks) lens[i].push_back(c->length); }
  }
  std::vector<std::shared_ptr<ArrayData>> results;
  if (kernel->can_execute_chunkwise) {
    // exec.go:152-155: "vector kernel arguments must all be the same length"
    int64_t l0 = args[0].Len();
    for (auto& a : args) if (a.Len() != l0) return Status::Invalid("vector kernel arguments must all be the same length");
    std::vector<SpanPiece> pieces;
    RETURN_NOT_OK(IterateExecSpans(lens, is_chunked, INT64_MAX, &pieces));
    if (pieces.empty()) { SpanPiece p; p.pos = 0; p.len = 0; p.chunk_index.assign(args.size(), 0); p.chunk_pos.assign(args.size(), 0); pieces.push_back(p); }
    for (auto& p : pieces) {
      ExecSpan span;
      span.len = p.len;
      span.values.assign(args.size(), ExecValue());
      for (size_t i = 0; i < args.size(); ++i) {
        if (args[i].kind == DatumKind::CHUNKED && args[i].chunked->chunks.empty()) { span.values[i].array.type = in_types[i]; continue; }
        const ArrayData& d = (args[i].kind == DatumKind::ARRAY) ? *args[i].array : *args[i].chunked->chunks[p.chunk_index[i]];
        span.values[i].array.SetMembers(d);
        span.values[i].array.SetSlice(d.offset + p.chunk_pos[i], p.len);
      }
      ArraySpan o;
      o.type = out_type;
      RETURN_NOT_OK(kernel->exec(&kctx, span, &o));
      results.push_back(o.MakeData());
    }
  } else if (have_chunked && kernel->exec_chunked && args.size() == 1) {
    ArraySpan o;
    o.type = out_type;
    RETURN_NOT_OK(kernel->exec_chunked(&kctx, *args[0].chunked, &o));
    results.push_back(o.MakeData());
  } else {
    if (have_chunked) return Status::NotImplemented("non-chunkwise vector kernel on chunked input (resolved by the meta function)");
    ExecSpan span;
    span.values.assign(args.size(), ExecValue());
    for (size_t i = 0; i < args.size(); ++i) span.values[i].array.SetMembers(*args[i].array);
    span.len = args.empty() ? 0 : args[0].array->length;
    ArraySpan o;
    o.type = out_type;
    RETURN_NOT_OK(kernel->exec(&kctx, span, &o));
    results.push_back(o.MakeData());
  }
  if (have_chunked) {
    auto c = std::make_shared<ChunkedArray>();
    c->type = out_type; c->chunks = results;
    for (auto& r : results) c->length += r->length;
    *out = Datum(c);
  } else {
    *out = Datum(results[0]);
  }
  return Status::OK();
}

Status CallFunction(const ExecCtx& ctx, const std::string& name, const FunctionOptions* opts, const std::vector<Datum>& args, Datum* out) {
  FunctionRegistry* reg = ctx.Registry ? ctx.Registry : GetFunctionRegistry();
  const Function* fn = reg->GetFunction(name);
  if (!fn) return Status::Make(AG_ERR_INVALID, "no function registered with name: " + name);  // arrow.ErrKey
  return fn->Execute(ctx, opts, args, out);
}

// ======================================================================================
// kernels (arrow/compute/internal/kernels) on device spans
// ======================================================================================
namespace {

using exec::ExecResult;

inline const uint8_t* ValuesPtr(const ArraySpan& a) {  // exec.GetSpanValues: Buf[1] advanced by Offset (exec/utils.go:38-44)
  return a.buffers[1].buf + a.offset * (BitWidth(a.type) / 8);
}
inline uint8_t* ValuesPtr(ExecResult* a) { return a->buffers[1].buf + a->offset * (BitWidth(a->type) / 8); }

const std::vector<Type>& kNumericTypesForCast() {
  static const std::vector<Type> v = {Type::UINT8, Type::INT8, Type::UINT16, Type::INT16, Type::UINT32, Type::INT32,
                                      Type::UINT64, Type::INT64, Type::FLOAT32, Type::FLOAT64};
  return v;
}

int ShapeOf(const ExecSpan& b) { return b.values[0].IsArray() ? (b.values[1].IsArray() ? AG_SHAPE_AA : AG_SHAPE_AS) : AG_SHAPE_SA; }

// ScalarBinary over the native loops (helpers.go:193-236 -> base_arithmetic_amd64.go:34-37)
exec::ArrayKernelExec ArithBinaryExec(int8_t op) {
  return [op](KernelCtx*, const ExecSpan& batch, ExecResult* out) -> Status {
    const int shape = ShapeOf(batch);
    const void* l = batch.values[0].IsArray() ? (const void*)ValuesPtr(batch.values[0].array) : (const void*)batch.values[0].scalar->value;
    const void* r = batch.values[1].IsArray() ? (const void*)ValuesPtr(batch.values[1].array) : (const void*)batch.values[1].scalar->value;
    NATIVE(ag_arith_binary_dev((int)out->type, op, shape, l, r, ValuesPtr(out), batch.len, nullptr));
    return Status::OK();
  };
}

// The same kernel over every aligned span of a chunked call in ONE launch
exec::BatchKernelExec ArithBinaryBatchExec(int8_t op) {
  return [op](KernelCtx*, const std::vector<ExecSpan>& spans, std::vector<ExecResult>& outs) -> Status {
    if (spans.empty()) return Status::OK();
    const int shape = ShapeOf(spans[0]);
    std::vector<ag_span3> table(spans.size());
    for (size_t i = 0; i < spans.size(); ++i) {
      const ExecValue &a = spans[i].values[0], &b = spans[i].values[1];
      table[i].l = a.IsArray() ? (const void*)ValuesPtr(a.array) : (const void*)a.scalar->value;
      table[i].r = b.IsArray() ? (const void*)ValuesPtr(b.array) : (const void*)b.scalar->value;
      table[i].out = ValuesPtr(&outs[i]);
      table[i].n = spans[i].len;
    }
    NATIVE(ag_arith_binary_spans_dev((int)outs[0].type, op, shape, table.data(), (int64_t)table.size(), nullptr));
    return Status::OK();
  };
}

// ScalarBinaryNotNull / checked integer kernels (helpers.go:284-380, base_arithmetic.go:249-294)
exec::ArrayKernelExec ArithCheckedExec(int8_t op) {
  return [op](KernelCtx* ctx, const ExecSpan& batch, ExecResult* out) -> Status {
    const int shape = ShapeOf(batch);
    const ExecValue &a = batch.values[0], &b = batch.values[1];
    // "fast path if one side is entirely null" (helpers.go:287): nothing is written
    if ((a.IsScalar() && !a.scalar->valid) || (b.IsScalar() && !b.scalar->valid)) return Status::OK();
    const void* l = a.IsArray() ? (const void*)a.array.buffers[1].buf : (const void*)a.scalar->value;
    const void* r = b.IsArray() ? (const void*)b.array.buffers[1].buf : (const void*)b.scalar->value;
    const int w = BitWidth(out->type) / 8;
    const uint8_t* lv = (a.IsArray() && a.array.MayHaveNulls()) ? a.array.buffers[0].buf : nullptr;
    const uint8_t* rv = (b.IsArray() && b.array.MayHaveNulls()) ? b.array.buffers[0].buf : nullptr;
    const int64_t loff = a.IsArray() ? a.array.offset : 0, roff = b.IsArray() ? b.array.offset : 0;
    if (a.IsArray()) l = (const uint8_t*)l + loff * w;
    if (b.IsArray()) r = (const uint8_t*)r + roff * w;
    NATIVE(ag_arith_checked_dev((int)out->type, op, shape, l, lv, loff, r, rv, roff, ValuesPtr(out), batch.len, ctx->error_word, nullptr));
    return Status::OK();
  };
}

// AbsoluteValueChecked / NegateChecked (base_arithmetic.go:295-340): every slot, MinInt -> "overflow"
exec::ArrayKernelExec ArithUnaryCheckedExec(int8_t op) {
  return [op](KernelCtx* ctx, const ExecSpan& batch, ExecResult* out) -> Status {
    NATIVE(ag_arith_unary_checked_dev((int)out->type, op, ValuesPtr(batch.values[0].array), ValuesPtr(out), batch.len, ctx->error_word, nullptr));
    return Status::OK();
  };
}

exec::ArrayKernelExec ArithUnaryExec(int8_t op) {
  return [op](KernelCtx*, const ExecSpan& batch, ExecResult* out) -> Status {
    NATIVE(ag_arith_unary_same_dev((int)out->type, op, ValuesPtr(batch.values[0].array), ValuesPtr(out), batch.len, nullptr));
    return Status::OK();
  };
}

// compareKernel (scalar_comparisons.go:199-218): output pointer at byte Offset/8, bit prefix Offset%8
exec::ArrayKernelExec CompareExec(int cmp) {
  return [cmp](KernelCtx*, const ExecSpan& batch, ExecResult* out) -> Status {
    const int shape = ShapeOf(batch);
    const ExecValue &a = batch.values[0], &b = batch.values[1];
    const void* l = a.IsArray() ? (const void*)ValuesPtr(a.array) : (const void*)a.scalar->value;
    const void* r = b.IsArray() ? (const void*)ValuesPtr(b.array) : (const void*)b.scalar->value;
    NATIVE(ag_compare_dev((int)a.type(), cmp, shape, l, r, out->buffers[1].buf + out->offset / 8, batch.len, (int)(out->offset % 8), nullptr));
    return Status::OK();
  };
}

// and / or / xor / and_not (scalar_boolean.go:67-279) incl. the scalar-operand special cases
exec::ArrayKernelExec BoolBinaryExec(int bitop) {
  return [bitop](KernelCtx*, const ExecSpan& batch, ExecResult* out) -> Status {
    const ExecValue &a = batch.values[0], &b = batch.values[1];
    uint8_t* ob = out->buffers[1].buf;
    if (a.IsArray() && b.IsArray()) {
      NATIVE(ag_bitmap_op_dev(bitop, a.array.buffers[1].buf, a.array.offset, b.array.buffers[1].buf, b.array.offset, ob, out->offset, batch.len, nullptr));
      return Status::OK();
    }
    // commutativeBinaryKernel / AndNot CallScalarLeft / CallScalarRight
    const bool scalar_left = a.IsScalar();
    const Scalar* s = scalar_left ? a.scalar : b.scalar;
    const ArraySpan& arr = scalar_left ? b.array : a.array;
    if (!s->valid) return Status::OK();
    bool sv = s->value[0] != 0;
    int op = bitop;
    if (bitop == AG_BITOP_ANDNOT && !scalar_left) { op = AG_BITOP_AND; sv = !sv; }  // AndNot.CallScalarRight = And with inverted scalar
    enum { COPY, INVERT, SET0, SET1 } act;
    switch (op) {
      case AG_BITOP_AND: act = sv ? COPY : SET0; break;
      case AG_BITOP_OR: act = sv ? SET1 : COPY; break;
      case AG_BITOP_XOR: act = sv ? INVERT : COPY; break;
      default: /* ANDNOT, scalar left */ act = sv ? INVERT : SET0; break;
    }
    switch (act) {
      case COPY: NATIVE(ag_bitmap_copy_dev(arr.buffers[1].buf, arr.offset, arr.len, ob, out->offset, nullptr)); break;
      case INVERT: NATIVE(ag_bitmap_invert_dev(arr.buffers[1].buf, arr.offset, arr.len, ob, out->offset, nullptr)); break;
      case SET0: NATIVE(ag_bitmap_set_dev(ob, out->offset, out->len, 0, nullptr)); break;
      case SET1: NATIVE(ag_bitmap_set_dev(ob, out->offset, out->len, 1, nullptr)); break;
    }
    return Status::OK();
  };
}

// Kleene and / or / and_not (scalar_boolean.go:92-334): array ⊕ array through computeKleene
// (:29-65); scalar operands through the CallScalarLeft tables (:109-141, :186-221, :296-330) with
// CallScalarRight = commutative swap (types.go:80-83), and_not's = and_kleene with the scalar
// inverted (:332-334).
exec::ArrayKernelExec KleeneExec(int kop, int plain_bitop) {
  return [kop, plain_bitop](KernelCtx*, const ExecSpan& batch, ExecResult* out) -> Status {
    if (batch.len == 0) return Status::OK();  // SimpleBinary, types.go:91-93
    const ExecValue &a = batch.values[0], &b = batch.values[1];
    uint8_t* ov = out->buffers[0].buf;
    uint8_t* od = out->buffers[1].buf;
    const int64_t oo = out->offset, n = batch.len;
    if (a.IsArray() && b.IsArray()) {
      ArraySpan l = a.array, r = b.array;
      int64_t ln = 0, rn = 0;
      RETURN_NOT_OK(l.UpdateNullCount(&ln));
      RETURN_NOT_OK(r.UpdateNullCount(&rn));
      if (ln == 0 && rn == 0) {
        NATIVE(ag_bitmap_set_dev(ov, oo, n, 1, nullptr));
        out->nulls = 0;
        NATIVE(ag_bitmap_op_dev(plain_bitop, l.buffers[1].buf, l.offset, r.buffers[1].buf, r.offset, od, oo, n, nullptr));
        return Status::OK();
      }
      NATIVE(ag_kleene_dev(kop, ln ? l.buffers[0].buf : nullptr, l.buffers[1].buf, l.offset, rn ? r.buffers[0].buf : nullptr, r.buffers[1].buf, r.offset,
                           ov, od, oo, n, nullptr));
      out->nulls = kUnknownNullCount;
      return Status::OK();
    }
    // one scalar operand.  Reduce to "scalar on the left" of a (possibly different) kernel.
    const bool scalar_left = a.IsScalar();
    const Scalar* sc = scalar_left ? a.scalar : b.scalar;
    ArraySpan arr = scalar_left ? b.array : a.array;
    bool s_valid = sc->valid, s_val = sc->value[0] != 0;
    int op = kop;  // which CallScalarLeft table to use
    if (kop == AG_KLEENE_ANDNOT && !scalar_left) { op = AG_KLEENE_AND; s_val = !s_val; }  // :332-334 (invertScalar keeps nulls)
    int64_t an = 0;
    RETURN_NOT_OK(arr.UpdateNullCount(&an));
    const uint8_t* av = arr.buffers[0].buf;
    const uint8_t* ad = arr.buffers[1].buf;
    const int64_t ao = arr.offset;
    auto all_valid = [&]() -> Status { NATIVE(ag_bitmap_set_dev(ov, oo, n, 1, nullptr)); out->nulls = 0; return Status::OK(); };
    auto copy_valid_from_arr = [&]() -> Status {
      if (an == 0) return all_valid();
      NATIVE(ag_bitmap_copy_dev(av, ao, n, ov, oo, nullptr));
      out->nulls = kUnknownNullCount;
      return Status::OK();
    };
    out->nulls = kUnknownNullCount;
    const bool s_true = s_valid && s_val, s_false = s_valid && !s_val;
    if (op == AG_KLEENE_AND) {          // KleeneAndOpKernel.CallScalarLeft :109-141
      if (s_false) { RETURN_NOT_OK(all_valid()); NATIVE(ag_bitmap_set_dev(od, oo, n, 0, nullptr)); }
      else if (s_true) { RETURN_NOT_OK(copy_valid_from_arr()); NATIVE(ag_bitmap_copy_dev(ad, ao, n, od, oo, nullptr)); }
      else {  // null scalar: valid iff right is (valid and) false
        if (an == 0) NATIVE(ag_bitmap_invert_dev(ad, ao, n, ov, oo, nullptr));
        else NATIVE(ag_bitmap_op_dev(AG_BITOP_ANDNOT, av, ao, ad, ao, ov, oo, n, nullptr));
        NATIVE(ag_bitmap_copy_dev(ad, ao, n, od, oo, nullptr));
      }
    } else if (op == AG_KLEENE_OR) {    // KleeneOrOpKernel.CallScalarLeft :186-221
      if (s_true) { RETURN_NOT_OK(all_valid()); NATIVE(ag_bitmap_set_dev(od, oo, n, 1, nullptr)); }
      else if (s_false) { RETURN_NOT_OK(copy_valid_from_arr()); NATIVE(ag_bitmap_copy_dev(ad, ao, n, od, oo, nullptr)); }
      else {  // null scalar: valid iff right is (valid and) true
        if (an == 0) NATIVE(ag_bitmap_copy_dev(ad, ao, n, ov, oo, nullptr));
        else NATIVE(ag_bitmap_op_dev(AG_BITOP_AND, av, ao, ad, ao, ov, oo, n, nullptr));
        NATIVE(ag_bitmap_copy_dev(ad, ao, n, od, oo, nullptr));
      }
    } else {                            // KleeneAndNotOpKernel.CallScalarLeft :296-330 (scalar AND NOT array)
      if (s_false) { RETURN_NOT_OK(all_valid()); NATIVE(ag_bitmap_set_dev(od, oo, n, 0, nullptr)); }
      else if (s_true) { RETURN_NOT_OK(copy_valid_from_arr()); NATIVE(ag_bitmap_invert_dev(ad, ao, n, od, oo, nullptr)); }
      else {  // null scalar: valid iff right is (valid and) true
        if (an == 0) NATIVE(ag_bitmap_copy_dev(ad, ao, n, ov, oo, nullptr));
        else NATIVE(ag_bitmap_op_dev(AG_BITOP_AND, av, ao, ad, ao, ov, oo, n, nullptr));
        NATIVE(ag_bitmap_invert_dev(ad, ao, n, od, oo, nullptr));
      }
    }
    return Status::OK();
  };
}

// isNullExec / isNotNullExec (scalar_comparisons.go:718-745): NullComputedNoPrealloc, MemNoPrealloc,
// the output never has a validity bitmap
Status IsNullExec(KernelCtx* ctx, const ExecSpan& batch, ExecResult* out) {
  const ArraySpan& in = batch.values[0].array;
  std::shared_ptr<Buffer> b;
  RETURN_NOT_OK(ctx->AllocateBitmap(in.len, &b));  // zero-filled: "no validity buffer" means all false
  if (in.buffers[0].buf) NATIVE(ag_bitmap_invert_dev(in.buffers[0].buf, in.offset, in.len, b->data(), 0, nullptr));
  out->type = Type::BOOL; out->len = in.len; out->offset = 0; out->nulls = 0;
  out->buffers[0] = exec::BufferSpan();
  out->buffers[1].buf = b->data(); out->buffers[1].len = b->size(); out->buffers[1].owner = b; out->buffers[1].self_alloc = true;
  return Status::OK();
}
Status IsNotNullExec(KernelCtx* ctx, const ExecSpan& batch, ExecResult* out) {
  const ArraySpan& in = batch.values[0].array;
  std::shared_ptr<Buffer> b;
  RETURN_NOT_OK(ctx->AllocateBitmap(in.len, &b));
  if (in.buffers[0].buf) NATIVE(ag_bitmap_copy_dev(in.buffers[0].buf, in.offset, in.len, b->data(), 0, nullptr));
  else NATIVE(ag_bitmap_set_dev(b->data(), 0, in.len, 1, nullptr));  // memory.Set(0xFF)
  out->type = Type::BOOL; out->len = in.len; out->offset = 0; out->nulls = 0;
  out->buffers[0] = exec::BufferSpan();
  out->buffers[1].buf = b->data(); out->buffers[1].len = b->size(); out->buffers[1].owner = b; out->buffers[1].self_alloc = true;
  return Status::OK();
}
// isNanKernelExec (scalar_comparisons.go:754-765): the NE kernel with the input on both sides;
// integer inputs are ConstBoolExec(false) (:747-752)
Status IsNanExec(KernelCtx*, const ExecSpan& batch, ExecResult* out) {
  const ArraySpan& in = batch.values[0].array;
  if (!IsFloating(in.type)) { NATIVE(ag_bitmap_set_dev(out->buffers[1].buf, out->offset, batch.len, 0, nullptr)); return Status::OK(); }
  NATIVE(ag_compare_dev((int)in.type, AG_CMP_NE, AG_SHAPE_AA, ValuesPtr(in), ValuesPtr(in), out->buffers[1].buf + out->offset / 8, batch.len,
                        (int)(out->offset % 8), nullptr));
  return Status::OK();
}

// NotExecKernel (scalar_boolean.go:336-347): invert data, share the validity buffer
// ---- numeric casts (kernels/numeric_cast.go:37-71 over cast_numeric.go:101-131) ----------
// Integer bounds of intsCanFit / checkIntToFloatTrunc, only needed to word the error like the
// reference ("integer value %d not in range: %d to %d", helpers.go:591-594).
void SafeIntBounds(Type in, Type out, __int128* lo, __int128* hi) {
  auto tmin = [](Type t) -> __int128 { return IsSignedInteger(t) ? -((__int128)1 << (BitWidth(t) - 1)) : 0; };
  auto tmax = [](Type t) -> __int128 { return IsSignedInteger(t) ? ((__int128)1 << (BitWidth(t) - 1)) - 1 : ((__int128)1 << BitWidth(t)) - 1; };
  if (IsFloating(out)) {
    const int mant = out == Type::FLOAT32 ? 24 : 53;
    *hi = (__int128)1 << mant;
    *lo = IsSignedInteger(in) ? -*hi : 0;
    return;
  }
  *lo = std::max(tmin(in), tmin(out));
  *hi = std::min(tmax(in), tmax(out));
}
std::string Int128ToString(__int128 v) {
  if (v == 0) return "0";
  const bool neg = v < 0;
  unsigned __int128 u = neg ? (unsigned __int128)(-(v + 1)) + 1 : (unsigned __int128)v;
  std::string r;
  while (u) { r.insert(r.begin(), (char)('0' + (int)(u % 10))); u /= 10; }
  return neg ? "-" + r : r;
}

Status CastNumericExec(KernelCtx* ctx, const ExecSpan& batch, ExecResult* out) {
  const auto* opts = static_cast<const CastOptions*>(ctx->state);
  const ArraySpan& in = batch.values[0].array;
  if (batch.len == 0) return Status::OK();
  NATIVE(ag_cast_numeric_checked_dev((int)in.type, (int)out->type, ValuesPtr(in), in.buffers[0].buf, in.offset, ValuesPtr(out), batch.len,
                                     opts->AllowIntOverflow ? 1 : 0, opts->AllowFloatTruncate ? 1 : 0, ctx->error_word, nullptr));
  // one 8-byte read per span: the error names the offending VALUE, like the reference's does
  int64_t bad = AG_NO_ERROR_POS;
  NATIVE(ag_download(&bad, ctx->error_word, sizeof(bad), nullptr));
  NATIVE(ag_stream_sync(nullptr));
  if (bad == AG_NO_ERROR_POS) return Status::OK();
  const int w = BitWidth(in.type) / 8;
  uint8_t raw[8] = {0};
  NATIVE(ag_download(raw, ValuesPtr(in) + bad * w, (size_t)w, nullptr));
  NATIVE(ag_stream_sync(nullptr));
  if (IsFloating(in.type)) {  // numeric_cast.go:614-617
    double v;
    if (in.type == Type::FLOAT32) { float f; memcpy(&f, raw, 4); v = f; } else memcpy(&v, raw, 8);
    char buf[128];
    snprintf(buf, sizeof(buf), "float value %f was truncated converting to %s", v, TypeName(out->type));
    return Status::Invalid(buf);
  }
  __int128 v = 0, lo, hi;
  switch (in.type) {
    case Type::INT8: v = (int8_t)raw[0]; break;
    case Type::UINT8: v = raw[0]; break;
    case Type::INT16: { int16_t t; memcpy(&t, raw, 2); v = t; break; }
    case Type::UINT16: { uint16_t t; memcpy(&t, raw, 2); v = t; break; }
    case Type::INT32: { int32_t t; memcpy(&t, raw, 4); v = t; break; }
    case Type::UINT32: { uint32_t t; memcpy(&t, raw, 4); v = t; break; }
    case Type::INT64: { int64_t t; memcpy(&t, raw, 8); v = t; break; }
    default: { uint64_t t; memcpy(&t, raw, 8); v = t; break; }
  }
  SafeIntBounds(in.type, out->type, &lo, &hi);
  return Status::Invalid("integer value " + Int128ToString(v) + " not in range: " + Int128ToString(lo) + " to " + Int128ToString(hi));
}

const char* CastFunctionName(Type t) {  // cast.go:841-880
  switch (t) {
    case Type::INT8: return "cast_int8"; case Type::INT16: return "cast_int16"; case Type::INT32: return "cast_int32";
    case Type::INT64: return "cast_int64"; case Type::UINT8: return "cast_uint8"; case Type::UINT16: return "cast_uint16";
    case Type::UINT32: return "cast_uint32"; case Type::UINT64: return "cast_uint64"; case Type::FLOAT32: return "cast_float";
    case Type::FLOAT64: return "cast_double"; default: return nullptr;
  }
}

std::shared_ptr<ScalarFunction> MakeCastTo(Type to) {  // GetCastToInteger / GetCastToFloating, numeric_cast.go:835-906
  auto fn = std::make_shared<ScalarFunction>(CastFunctionName(to), 1);
  for (Type t : kNumericTypesForCast()) {
    exec::ScalarKernel k;
    k.in_types = {t};
    k.out_type = [to](const std::vector<Type>&) { return to; };
    k.exec = CastNumericExec;
    k.can_fail = true;  // the executor supplies the error word; CastNumericExec words the error itself
    k.fail_message = "cast failed";
    fn->AddKernel(std::move(k));
  }
  return fn;
}

Status NotExec(KernelCtx*, const ExecSpan& batch, ExecResult* out) {
  const ArraySpan& in = batch.values[0].array;
  NATIVE(ag_bitmap_invert_dev(in.buffers[1].buf, in.offset, in.len, out->buffers[1].buf, out->offset, nullptr));
  if (in.buffers[0].buf && in.nulls != 0) {
    if (in.offset == out->offset) { out->buffers[0] = in.buffers[0]; out->buffers[0].self_alloc = false; }
    else {
      std::shared_ptr<Buffer> b;
      RETURN_NOT_OK(Buffer::Allocate((out->offset + out->len + 7) / 8, &b));
      NATIVE(ag_bitmap_copy_dev(in.buffers[0].buf, in.offset, in.len, b->data(), out->offset, nullptr));
      out->buffers[0].buf = b->data(); out->buffers[0].len = b->size(); out->buffers[0].owner = b; out->buffers[0].self_alloc = true;
    }
  }
  out->nulls = in.nulls;
  return Status::OK();
}

// PrimitiveFilter (vector_selection.go:449-520)
Status PrimitiveFilterExec(KernelCtx* ctx, const ExecSpan& batch, ExecResult* out) {
  ArraySpan values = batch.values[0].array, filter = batch.values[1].array;
  const FilterOptions* opts = static_cast<const FilterOptions*>(ctx->state);
  const int sel = opts ? (int)opts->NullSelection : (int)DropNulls;
  int64_t vn = 0, fn = 0;
  RETURN_NOT_OK(values.UpdateNullCount(&vn));
  RETURN_NOT_OK(filter.UpdateNullCount(&fn));
  const uint8_t* mvalid = fn != 0 ? filter.buffers[0].buf : nullptr;
  const uint8_t* vvalid = vn != 0 ? values.buffers[0].buf : nullptr;
  // getFilterOutputSize (:57-81)
  std::shared_ptr<Buffer> scal;
  RETURN_NOT_OK(Buffer::Allocate(16, &scal));
  NATIVE(ag_filter_output_size_dev(filter.buffers[1].buf, mvalid, filter.offset, filter.len, sel, (int64_t*)scal->data(), nullptr));
  int64_t out_len = 0;
  RETURN_NOT_OK(scal->ToHost(&out_len, 8));
  out->nulls = (vn == 0 && (sel == DropNulls || fn == 0)) ? 0 : kUnknownNullCount;  // :464-468
  const bool allocate_validity = vn != 0 || fn != 0;                                  // :473
  const int bw = BitWidth(values.type);
  // preallocateData (:83-93)
  out->type = values.type; out->len = out_len; out->offset = 0;
  std::shared_ptr<Buffer> data, valid;
  RETURN_NOT_OK(ctx->Allocate(bw == 1 ? ((out_len + 31) / 32) * 4 : out_len * (bw / 8), &data));
  out->buffers[1].buf = data->data(); out->buffers[1].len = data->size(); out->buffers[1].owner = data; out->buffers[1].self_alloc = true;
  if (allocate_validity) {
    RETURN_NOT_OK(ctx->Allocate(((out_len + 31) / 32) * 4, &valid));
    out->buffers[0].buf = valid->data(); out->buffers[0].len = valid->size(); out->buffers[0].owner = valid; out->buffers[0].self_alloc = true;
  }
  if (values.len == 0) return Status::OK();
  NATIVE(ag_filter_primitive_dev(bw, values.buffers[1].buf, vvalid, values.offset, filter.buffers[1].buf, mvalid, filter.offset, values.len, sel,
                                 data->data(), allocate_validity ? valid->data() : nullptr, out_len, (int64_t*)scal->data() + 1, nullptr));
  return Status::OK();
}

// ---- cumulative_sum[_checked] (kernels/vector_cumulative.go:332-410) -------------------------
// cumulativeStartValue :81-112: nil -> zero, null scalar -> error, other types -> safe cast.
Status CumulativeStart(const CumulativeOptions* opts, Type t, bool* has_start, uint8_t (&raw)[8]) {
  *has_start = false;
  memset(raw, 0, 8);
  if (!opts || !opts->Start) return Status::OK();
  if (!opts->Start->valid) return Status::Invalid("cumulative sum start value must be valid");
  std::shared_ptr<Scalar> sc = opts->Start;
  if (sc->type != t) {
    Datum casted;
    ExecCtx ectx;
    Status st = CastDatum(ectx, Datum(sc), SafeCastOptions(t), &casted);
    if (!st.ok()) return Status::Invalid(std::string("cannot cast cumulative sum start value to ") + TypeName(t) + ": " + st.msg);
    sc = casted.scalar;
  }
  memcpy(raw, sc->value, 8);
  *has_start = true;
  return Status::OK();
}

struct CumsumRun {  // device state + error word shared by the chunks of one call
  std::shared_ptr<Buffer> state, bad;
  Status Init(Type t, const CumulativeOptions* opts) {
    bool has_start; uint8_t raw[8];
    RETURN_NOT_OK(CumulativeStart(opts, t, &has_start, raw));
    RETURN_NOT_OK(Buffer::Allocate(sizeof(ag_cumsum_state), &state));
    RETURN_NOT_OK(Buffer::Allocate(8, &bad));
    NATIVE(ag_cumulative_sum_state_init_dev(state->data(), (int)t, has_start ? raw : nullptr, nullptr));
    NATIVE(ag_error_word_reset_dev((int64_t*)bad->data(), nullptr));
    return Status::OK();
  }
};

// cumulativeSumSpans: one output array for all input spans; validity only when some span may have nulls
Status CumulativeSpans(bool checked, const CumulativeOptions* opts, Type t, const std::vector<ArraySpan>& inputs, ExecResult* out) {
  if (!IsInteger(t) && !IsFloating(t)) return Status::TypeError(std::string("cumulative sum input type must be numeric, got ") + TypeName(t));
  int64_t total = 0;
  bool needs_validity = false;
  for (auto& in : inputs) { total += in.len; needs_validity = needs_validity || (in.buffers[0].buf != nullptr && in.nulls != 0); }
  out->type = t; out->len = total; out->offset = 0; out->nulls = 0;
  if (total == 0) return Status::OK();
  CumsumRun run;
  RETURN_NOT_OK(run.Init(t, opts));
  std::shared_ptr<Buffer> data, validity;
  const int w = BitWidth(t) / 8;
  RETURN_NOT_OK(Buffer::Allocate(total * w, &data));
  if (needs_validity) RETURN_NOT_OK(Buffer::Allocate(BytesForBits(total), &validity));
  int64_t pos = 0;
  for (auto& in : inputs) {
    if (in.len == 0) continue;
    // a bitmap that is known to be all set (null_count == 0: Array.from_numpy(valid=all true), filter / take outputs,
    // preallocated PropagateNulls bitmaps) takes the no-nulls path like the reference (vector_cumulative.go:341-346)
    const uint8_t* in_valid = in.nulls != 0 ? in.buffers[0].buf : nullptr;
    NATIVE(ag_cumulative_sum_dev((int)t, ValuesPtr(in), in_valid, in.offset, in.len, opts && opts->SkipNulls ? 1 : 0, checked ? 1 : 0,
                                 data->data() + pos * w, validity ? validity->data() : nullptr, pos, run.state->data(), (int64_t*)run.bad->data(), nullptr));
    pos += in.len;
  }
  if (checked) {
    int64_t bad = 0;
    RETURN_NOT_OK(run.bad->ToHost(&bad, 8));
    if (bad != AG_NO_ERROR_POS) return Status::Invalid("overflow");  // errOverflow, base_arithmetic.go:137
  }
  out->buffers[1].buf = data->data(); out->buffers[1].len = data->size(); out->buffers[1].owner = data;
  if (validity) {
    ag_cumsum_state hs;
    RETURN_NOT_OK(run.state->ToHost(&hs, sizeof(hs)));
    out->buffers[0].buf = validity->data(); out->buffers[0].len = validity->size(); out->buffers[0].owner = validity;
    out->nulls = hs.null_count;
  }
  return Status::OK();
}

exec::ArrayKernelExec CumulativeExec(bool checked) {  // cumulativeSumExec :370-383
  return [checked](KernelCtx* ctx, const ExecSpan& batch, ExecResult* out) -> Status {
    const ArraySpan& in = batch.values[0].array;
    return CumulativeSpans(checked, static_cast<const CumulativeOptions*>(ctx->state), in.type, {in}, out);
  };
}

std::function<Status(KernelCtx*, const ChunkedArray&, ExecResult*)> CumulativeExecChunked(bool checked) {  // :385-410
  return [checked](KernelCtx* ctx, const ChunkedArray& c, ExecResult* out) -> Status {
    std::vector<ArraySpan> spans(c.chunks.size());
    for (size_t i = 0; i < c.chunks.size(); ++i) spans[i].SetMembers(*c.chunks[i]);
    return CumulativeSpans(checked, static_cast<const CumulativeOptions*>(ctx->state), c.type, spans, out);
  };
}

std::shared_ptr<VectorFunction> MakeCumulative(const std::string& name, bool checked) {
  auto fn = std::make_shared<VectorFunction>(name, 1);
  exec::VectorKernel k;
  k.any_input_type = true;  // the exec rejects non-numeric inputs with ErrType like the reference's start-value check
  k.out_type = [](const std::vector<Type>& t) { return t[0]; };
  k.exec = CumulativeExec(checked);
  k.exec_chunked = CumulativeExecChunked(checked);
  k.null_handling = exec::NullHandling::COMPUTED_NO_PREALLOC;
  k.mem_alloc = exec::MemAlloc::NO_PREALLOC;
  k.can_execute_chunkwise = false;  // vector_cumulative.go:420-421
  fn->AddKernel(std::move(k));
  return fn;
}

// PrimitiveTake (vector_selection.go:1162-1192)
Status PrimitiveTakeExec(KernelCtx* ctx, const ExecSpan& batch, ExecResult* out) {
  ArraySpan values = batch.values[0].array, indices = batch.values[1].array;
  const TakeOptions* opts = static_cast<const TakeOptions*>(ctx->state);
  const bool bounds = opts ? opts->BoundsCheck : true;
  if (!IsInteger(indices.type)) return Status::Invalid("invalid index type for bounds checking");  // helpers.go:978
  int64_t vn = 0, in_ = 0;
  RETURN_NOT_OK(values.UpdateNullCount(&vn));
  RETURN_NOT_OK(indices.UpdateNullCount(&in_));
  const int bw = BitWidth(values.type);
  const bool allocate_validity = vn != 0 || in_ != 0;  // :1175
  out->type = values.type; out->len = indices.len; out->offset = 0;
  std::shared_ptr<Buffer> data, valid, word;
  RETURN_NOT_OK(ctx->Allocate(bw == 1 ? ((indices.len + 31) / 32) * 4 : indices.len * (bw / 8), &data));
  out->buffers[1].buf = data->data(); out->buffers[1].len = data->size(); out->buffers[1].owner = data; out->buffers[1].self_alloc = true;
  if (allocate_validity) {
    RETURN_NOT_OK(ctx->Allocate(((indices.len + 31) / 32) * 4, &valid));
    out->buffers[0].buf = valid->data(); out->buffers[0].len = valid->size(); out->buffers[0].owner = valid; out->buffers[0].self_alloc = true;
  }
  out->nulls = allocate_validity ? kUnknownNullCount : 0;
  if (indices.len == 0) return Status::OK();
  RETURN_NOT_OK(Buffer::Allocate(8, &word));
  NATIVE(ag_error_word_reset_dev((int64_t*)word->data(), nullptr));
  const int iw = BitWidth(indices.type);
  NATIVE(ag_take_primitive_dev(bw, values.buffers[1].buf, vn ? values.buffers[0].buf : nullptr, values.offset, values.len, iw, IsSignedInteger(indices.type),
                               indices.buffers[1].buf + indices.offset * (iw / 8), in_ ? indices.buffers[0].buf : nullptr, indices.offset, indices.len,
                               bounds ? 1 : 0, data->data(), allocate_validity ? valid->data() : nullptr, (int64_t*)word->data(), nullptr));
  if (bounds) {
    int64_t bad = 0;
    RETURN_NOT_OK(word->ToHost(&bad, 8));
    if (bad != AG_NO_ERROR_POS) {
      // "%d out of bounds" with the offending index value (helpers.go:951)
      uint8_t raw[8] = {0};
      RETURN_NOT_OK(indices.buffers[1].owner->ToHost(raw, iw / 8, (indices.offset + bad) * (iw / 8)));
      long long v = 0; unsigned long long uv = 0;
      memcpy(&uv, raw, 8);
      if (IsSignedInteger(indices.type)) {
        switch (iw) { case 8: v = (int8_t)raw[0]; break; case 16: { int16_t t; memcpy(&t, raw, 2); v = t; break; }
                      case 32: { int32_t t; memcpy(&t, raw, 4); v = t; break; } default: memcpy(&v, raw, 8); }
        return Status::IndexError(std::to_string(v) + " out of bounds");
      }
      return Status::IndexError(std::to_string(uv) + " out of bounds");
    }
  }
  return Status::OK();
}

Type FirstType(const std::vector<Type>& t) { return t[0]; }
Type BoolType(const std::vector<Type>&) { return Type::BOOL; }

const Type kNumericTypes[] = {Type::UINT8, Type::INT8, Type::UINT16, Type::INT16, Type::UINT32, Type::INT32, Type::UINT64, Type::INT64, Type::FLOAT32, Type::FLOAT64};

std::shared_ptr<ScalarFunction> MakeArithBinary(const std::string& name, int8_t unchecked_op, int8_t checked_op, bool checked, const char* fail_msg) {
  // GetArithmeticBinaryKernels (scalar_arithmetic.go:86-95): one [ty,ty]->ty kernel per numeric type
  auto fn = std::make_shared<ScalarFunction>(name, 2);
  fn->promote_numeric = true;  // arithmeticFunction.DispatchBest, arithmetic.go:112-140
  for (Type t : kNumericTypes) {
    exec::ScalarKernel k;
    k.in_types = {t, t};
    k.out_type = FirstType;
    if (checked && IsInteger(t)) {  // integral checked funcs use the NotNull versions (base_arithmetic_amd64.go:103-106)
      k.exec = ArithCheckedExec(checked_op);
      k.can_fail = true;
      k.fail_message = fail_msg;
    } else {
      k.exec = ArithBinaryExec(checked ? checked_op : unchecked_op);
      k.exec_batch = ArithBinaryBatchExec(checked ? checked_op : unchecked_op);
    }
    fn->AddKernel(std::move(k));
  }
  return fn;
}

// divide / divide_unchecked (arithmetic.go:782-785; kernels base_arithmetic.go:154-161,287-294,386-397): every kernel is
// ScalarBinaryNotNull.  Integers fail on a zero divisor in BOTH flavours; floats only in the checked one.
std::shared_ptr<ScalarFunction> MakeDivide(const std::string& name, bool checked) {
  auto fn = std::make_shared<ScalarFunction>(name, 2);
  fn->promote_numeric = true;
  for (Type t : kNumericTypes) {
    exec::ScalarKernel k;
    k.in_types = {t, t};
    k.out_type = FirstType;
    k.exec = ArithCheckedExec(checked ? AG_OP_DIV_CHECKED : AG_OP_DIV);
    k.can_fail = true;   // the NotNull entry point always takes an error word; the unchecked float op never raises it
    k.fail_message = "divide by zero";
    fn->AddKernel(std::move(k));
  }
  return fn;
}

const Type kIntTypes[] = {Type::UINT8, Type::INT8, Type::UINT16, Type::INT16, Type::UINT32, Type::INT32, Type::UINT64, Type::INT64};

// bit_wise_and / or / xor (arithmetic.go:944-961, GetBitwiseBinaryKernels scalar_arithmetic.go:245-255): integer types,
// every slot; validity by intersection
std::shared_ptr<ScalarFunction> MakeBitwiseBinary(const std::string& name, int8_t op) {
  auto fn = std::make_shared<ScalarFunction>(name, 2);
  fn->promote_numeric = true;
  for (Type t : kIntTypes) {
    exec::ScalarKernel k;
    k.in_types = {t, t};
    k.out_type = FirstType;
    k.exec = ArithBinaryExec(op);
    k.exec_batch = ArithBinaryBatchExec(op);
    fn->AddKernel(std::move(k));
  }
  return fn;
}

// shift_left / shift_right (+ _unchecked) (arithmetic.go:970-996, GetShiftKernels scalar_arithmetic.go:401-412)
std::shared_ptr<ScalarFunction> MakeShift(const std::string& name, int8_t op, bool checked) {
  auto fn = std::make_shared<ScalarFunction>(name, 2);
  fn->promote_numeric = true;
  for (Type t : kIntTypes) {
    exec::ScalarKernel k;
    k.in_types = {t, t};
    k.out_type = FirstType;
    k.exec = ArithCheckedExec(op);
    k.can_fail = true;   // error word always supplied; only the checked ops raise it
    k.fail_message = "shift amount must be >= 0 and less than precision of type";
    fn->AddKernel(std::move(k));
  }
  return fn;
}

std::shared_ptr<ScalarFunction> MakeArithUnary(const std::string& name, int8_t op) {
  auto fn = std::make_shared<ScalarFunction>(name, 1);
  for (Type t : kNumericTypes) {
    exec::ScalarKernel k;
    k.in_types = {t};
    k.out_type = FirstType;
    k.exec = ArithUnaryExec(op);
    fn->AddKernel(std::move(k));
  }
  return fn;
}

std::shared_ptr<ScalarFunction> MakeArithUnaryChecked(const std::string& name, int8_t op, bool signed_only) {
  auto fn = std::make_shared<ScalarFunction>(name, 1);
  for (Type t : kNumericTypes) {
    if (signed_only && !IsSignedInteger(t) && !IsFloating(t)) continue;  // GetArithmeticUnarySignedKernels, arithmetic.go:839-840
    exec::ScalarKernel k;
    k.in_types = {t};
    k.out_type = FirstType;
    if (IsSignedInteger(t)) { k.exec = ArithUnaryCheckedExec(op); k.can_fail = true; k.fail_message = "overflow"; }
    else k.exec = ArithUnaryExec(op);
    fn->AddKernel(std::move(k));
  }
  return fn;
}

std::shared_ptr<ScalarFunction> MakeCompare(const std::string& name, int cmp) {  // CompareKernels, scalar_comparisons.go:654-716
  auto fn = std::make_shared<ScalarFunction>(name, 2);
  fn->promote_numeric = true;  // compareFunction.DispatchBest, scalar_compare.go:37-65
  for (Type t : kNumericTypes) {
    exec::ScalarKernel k;
    k.in_types = {t, t};
    k.out_type = BoolType;
    k.exec = CompareExec(cmp);
    fn->AddKernel(std::move(k));
  }
  return fn;
}

std::shared_ptr<ScalarFunction> MakeBool(const std::string& name, exec::ArrayKernelExec ex, exec::NullHandling nh) {  // scalar_bool.go:123-140
  auto fn = std::make_shared<ScalarFunction>(name, 2);
  exec::ScalarKernel k;
  k.in_types = {Type::BOOL, Type::BOOL};
  k.out_type = BoolType;
  k.exec = std::move(ex);
  k.null_handling = nh;
  fn->AddKernel(std::move(k));
  return fn;
}

Status ConcatenateChunks(const ChunkedArray& c, std::shared_ptr<ArrayData>* out);
Status DictionaryEncodeImpl(const DictionaryEncodeOptions& opts, const Datum& values, Datum* out);

}  // namespace

// GetFunctionRegistry (registry.go:47-62): the functions of the hot path under their reference names
FunctionRegistry* GetFunctionRegistry() {
  static FunctionRegistry* reg = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    reg = new FunctionRegistry();
    // arithmetic.go:635-636,679-682,782-785: add / sub / multiply (+ "subtract" alias) and _unchecked
    reg->AddFunction(MakeArithBinary("add", AG_OP_ADD, AG_OP_ADD_CHECKED, true, "overflow"), false);
    reg->AddFunction(MakeArithBinary("add_unchecked", AG_OP_ADD, AG_OP_ADD_CHECKED, false, ""), false);
    reg->AddFunction(MakeArithBinary("sub", AG_OP_SUB, AG_OP_SUB_CHECKED, true, "overflow"), false);
    reg->AddFunction(MakeArithBinary("sub_unchecked", AG_OP_SUB, AG_OP_SUB_CHECKED, false, ""), false);
    reg->AddAlias("subtract", "sub");
    reg->AddAlias("subtract_unchecked", "sub_unchecked");
    reg->AddFunction(MakeArithBinary("multiply", AG_OP_MUL, AG_OP_MUL_CHECKED, true, "overflow"), false);
    reg->AddFunction(MakeArithBinary("multiply_unchecked", AG_OP_MUL, AG_OP_MUL_CHECKED, false, ""), false);
    reg->AddFunction(MakeArithUnary("abs_unchecked", AG_OP_ABS), false);
    reg->AddFunction(MakeArithUnary("negate_unchecked", AG_OP_NEGATE), false);
    reg->AddFunction(MakeArithUnary("sign", AG_OP_SIGN), false);
    reg->AddFunction(MakeArithUnaryChecked("abs", AG_OP_ABS_CHECKED, false), false);       // arithmetic.go:822-823
    reg->AddFunction(MakeArithUnaryChecked("negate", AG_OP_NEGATE_CHECKED, true), false);  // arithmetic.go:839-846
    reg->AddFunction(MakeDivide("divide", true), false);                                   // arithmetic.go:784-785
    reg->AddFunction(MakeDivide("divide_unchecked", false), false);
    reg->AddFunction(MakeBitwiseBinary("bit_wise_and", AG_OP_BIT_AND), false);             // arithmetic.go:949-951
    reg->AddFunction(MakeBitwiseBinary("bit_wise_or", AG_OP_BIT_OR), false);
    reg->AddFunction(MakeBitwiseBinary("bit_wise_xor", AG_OP_BIT_XOR), false);
    {
      auto fn = std::make_shared<ScalarFunction>("bit_wise_not", 1);                       // arithmetic.go:965-972
      for (Type t : kIntTypes) {
        exec::ScalarKernel k;
        k.in_types = {t};
        k.out_type = FirstType;
        k.exec = ArithUnaryExec(AG_OP_BIT_NOT);
        fn->AddKernel(std::move(k));
      }
      reg->AddFunction(fn, false);
    }
    reg->AddFunction(MakeShift("shift_left", AG_OP_SHIFT_LEFT_CHECKED, true), false);      // arithmetic.go:980-983
    reg->AddFunction(MakeShift("shift_left_unchecked", AG_OP_SHIFT_LEFT, false), false);
    reg->AddFunction(MakeShift("shift_right", AG_OP_SHIFT_RIGHT_CHECKED, true), false);
    reg->AddFunction(MakeShift("shift_right_unchecked", AG_OP_SHIFT_RIGHT, false), false);
    // scalar_compare.go:102-153
    reg->AddFunction(MakeCompare("equal", AG_CMP_EQ), false);
    reg->AddFunction(MakeCompare("not_equal", AG_CMP_NE), false);
    reg->AddFunction(MakeCompare("greater", AG_CMP_GT), false);
    reg->AddFunction(MakeCompare("greater_equal", AG_CMP_GE), false);
    reg->AddFunction(MakeCompare("less", AG_CMP_LT), false);
    reg->AddFunction(MakeCompare("less_equal", AG_CMP_LE), false);
    // scalar_bool.go:123-140
    reg->AddFunction(MakeBool("and", BoolBinaryExec(AG_BITOP_AND), exec::NullHandling::INTERSECTION), false);
    reg->AddFunction(MakeBool("or", BoolBinaryExec(AG_BITOP_OR), exec::NullHandling::INTERSECTION), false);
    reg->AddFunction(MakeBool("xor", BoolBinaryExec(AG_BITOP_XOR), exec::NullHandling::INTERSECTION), false);
    reg->AddFunction(MakeBool("and_not", BoolBinaryExec(AG_BITOP_ANDNOT), exec::NullHandling::INTERSECTION), false);
    reg->AddFunction(MakeBool("and_kleene", KleeneExec(AG_KLEENE_AND, AG_BITOP_AND), exec::NullHandling::COMPUTED_PREALLOC), false);
    reg->AddFunction(MakeBool("or_kleene", KleeneExec(AG_KLEENE_OR, AG_BITOP_OR), exec::NullHandling::COMPUTED_PREALLOC), false);
    reg->AddFunction(MakeBool("and_not_kleene", KleeneExec(AG_KLEENE_ANDNOT, AG_BITOP_ANDNOT), exec::NullHandling::COMPUTED_PREALLOC), false);
    {
      auto fn = std::make_shared<ScalarFunction>("not", 1);
      exec::ScalarKernel k;
      k.in_types = {Type::BOOL};
      k.out_type = BoolType;
      k.exec = NotExec;
      k.null_handling = exec::NullHandling::COMPUTED_NO_PREALLOC;
      k.can_write_into_slices = false;
      fn->AddKernel(std::move(k));
      reg->AddFunction(fn, false);
    }
    // scalar_compare.go / scalar_comparisons.go:718-813: is_null, is_not_null, is_nan
    for (auto& spec : std::vector<std::pair<const char*, exec::ArrayKernelExec>>{{"is_null", IsNullExec}, {"is_not_null", IsNotNullExec}}) {
      auto fn = std::make_shared<ScalarFunction>(spec.first, 1);
      exec::ScalarKernel k;
      k.any_input_type = true;
      k.out_type = BoolType;
      k.exec = spec.second;
      k.null_handling = exec::NullHandling::COMPUTED_NO_PREALLOC;
      k.mem_alloc = exec::MemAlloc::NO_PREALLOC;
      k.can_write_into_slices = false;
      fn->AddKernel(std::move(k));
      reg->AddFunction(fn, false);
    }
    {
      auto fn = std::make_shared<ScalarFunction>("is_nan", 1);
      for (Type t : kNumericTypes) {
        exec::ScalarKernel k;
        k.in_types = {t};
        k.out_type = BoolType;
        k.exec = IsNanExec;
        k.null_handling = exec::NullHandling::OUTPUT_NOT_NULL;
        fn->AddKernel(std::move(k));
      }
      reg->AddFunction(fn, false);
    }
    // cast.go:45-81,841-880: cast_<type> scalar functions for the numeric types + the "cast" meta function
    for (Type t : kNumericTypes) reg->AddFunction(MakeCastTo(t), false);
    reg->AddFunction(std::make_shared<MetaFunction>("cast", 1, [](const ExecCtx& ctx, const FunctionOptions* fo, const std::vector<Datum>& args, Datum* out) -> Status {
      const auto* co = dynamic_cast<const CastOptions*>(fo);
      if (!co || co->ToType == Type::NA) return Status::Invalid("cast requires that options be passed with a ToType");
      if (args.size() != 1 || args[0].kind == DatumKind::NONE) return Status::Invalid("cast takes one value argument");
      RETURN_NOT_OK(RejectDictionaries("cast", args));
      if (args[0].type() == co->ToType) { *out = args[0]; return Status::OK(); }
      const char* fname = CastFunctionName(co->ToType);
      FunctionRegistry* r = ctx.Registry ? ctx.Registry : GetFunctionRegistry();
      const Function* fn = fname ? r->GetFunction(fname) : nullptr;
      if (!fn) return Status::NotImplemented(std::string("unsupported cast to ") + TypeName(co->ToType) + " from " + TypeName(args[0].type()));
      if (args[0].kind != DatumKind::SCALAR) return fn->Execute(ctx, fo, args, out);
      // scalar input: a one-element array through the same kernel (the reference promotes scalars to
      // length-1 arrays for scalar-only execution too, executor.go PromoteExecSpanScalars)
      const Scalar& sc = *args[0].scalar;
      auto res = std::make_shared<Scalar>();
      res->type = co->ToType;
      if (!sc.valid) { *out = Datum(res); return Status::OK(); }
      std::shared_ptr<ArrayData> one;
      RETURN_NOT_OK(ArrayData::FromHost(sc.type, 1, 0, nullptr, sc.value, 0, &one));
      Datum casted;
      RETURN_NOT_OK(fn->Execute(ctx, fo, {Datum(one)}, &casted));
      RETURN_NOT_OK(casted.array->ToHost(res->value, nullptr, nullptr));
      res->valid = true;
      *out = Datum(res);
      return Status::OK();
    }), false);
    // vector_sort.go:383-390, vector_hash.go, scalar_set_lookup.go: registry names bound to the GPU kernels
    reg->AddFunction(std::make_shared<MetaFunction>("sort_indices", 1, [](const ExecCtx& ctx, const FunctionOptions* fo, const std::vector<Datum>& args, Datum* out) -> Status {
      const auto* so = dynamic_cast<const SortOptions*>(fo);
      if (args.size() != 1) return Status::Invalid("sort_indices takes one argument");
      return SortIndices(ctx, args[0], so ? *so : SortOptions(), out);
    }), false);
    reg->AddFunction(std::make_shared<MetaFunction>("unique", 1, [](const ExecCtx& ctx, const FunctionOptions*, const std::vector<Datum>& args, Datum* out) -> Status {
      if (args.size() != 1) return Status::Invalid("unique takes one argument");
      return Unique(ctx, args[0], out);
    }), false);
    reg->AddFunction(std::make_shared<MetaFunction>("is_in", 1, [](const ExecCtx& ctx, const FunctionOptions* fo, const std::vector<Datum>& args, Datum* out) -> Status {
      const auto* so = dynamic_cast<const SetLookupOptions*>(fo);
      if (!so) return Status::Invalid("is_in requires SetLookupOptions");
      if (args.size() != 1) return Status::Invalid("is_in takes one argument");
      return IsIn(ctx, *so, args[0], out);
    }), false);
    reg->AddFunction(std::make_shared<MetaFunction>("dictionary_encode", 1, [](const ExecCtx& ctx, const FunctionOptions* fo, const std::vector<Datum>& args, Datum* out) -> Status {
      const auto* o = dynamic_cast<const DictionaryEncodeOptions*>(fo);
      if (args.size() != 1) return Status::Invalid("dictionary_encode takes one argument");
      return DictionaryEncodeImpl(o ? *o : DictionaryEncodeOptions(), args[0], out);
    }), false);
    // vector_cumulative.go:75-93
    reg->AddFunction(MakeCumulative("cumulative_sum", false), false);
    reg->AddFunction(MakeCumulative("cumulative_sum_checked", true), false);
    // selection.go:593-650: array_filter / array_take vector functions + filter / take meta functions
    {
      auto fn = std::make_shared<VectorFunction>("array_filter", 2);
      exec::VectorKernel k;
      k.any_input_type = true;
      k.out_type = FirstType;
      k.exec = PrimitiveFilterExec;
      k.null_handling = exec::NullHandling::COMPUTED_NO_PREALLOC;
      k.mem_alloc = exec::MemAlloc::NO_PREALLOC;
      k.can_execute_chunkwise = true;
      fn->AddKernel(std::move(k));
      reg->AddFunction(fn, false);
    }
    {
      auto fn = std::make_shared<VectorFunction>("array_take", 2);
      exec::VectorKernel k;
      k.any_input_type = true;
      k.out_type = FirstType;
      k.exec = PrimitiveTakeExec;
      k.null_handling = exec::NullHandling::COMPUTED_NO_PREALLOC;
      k.mem_alloc = exec::MemAlloc::NO_PREALLOC;
      k.can_execute_chunkwise = false;  // selection.go:639
      fn->AddKernel(std::move(k));
      reg->AddFunction(fn, false);
    }
    reg->AddFunction(std::make_shared<MetaFunction>("filter", 2, [](const ExecCtx& ctx, const FunctionOptions* opts, const std::vector<Datum>& args, Datum* out) -> Status {
      // filterMetaFunc, selection.go:41-85
      if (args.size() != 2) return Status::Invalid("filter takes 2 arguments");
      if (args[1].kind != DatumKind::ARRAY && args[1].kind != DatumKind::CHUNKED) return Status::NotImplemented("filter should be array-like");
      if (args[1].type() != Type::BOOL) return Status::NotImplemented("filter argument must be boolean type");
      return CallFunction(ctx, "array_filter", opts, args, out);
    }), false);
    reg->AddFunction(std::make_shared<MetaFunction>("take", 2, [](const ExecCtx& ctx, const FunctionOptions* opts, const std::vector<Datum>& args, Datum* out) -> Status {
      // takeMetaFunc, selection.go:93-114 -> takeArrayImpl :206-244 / takeChunkedImpl :246-300
      if (args.size() != 2) return Status::Invalid("take takes 2 arguments");
      RETURN_NOT_OK(RejectDictionaries("take", args));
      if (args[1].kind != DatumKind::ARRAY && args[1].kind != DatumKind::CHUNKED) return Status::NotImplemented("unsupported types for take operation");
      Datum values = args[0];
      const bool values_chunked = values.kind == DatumKind::CHUNKED;
      if (values_chunked) {  // ChunkedPrimitiveTake resolves chunks per index; on the device we gather from one table
        std::shared_ptr<ArrayData> cat;
        RETURN_NOT_OK(ConcatenateChunks(*values.chunked, &cat));
        values = Datum(cat);
      } else if (values.kind != DatumKind::ARRAY) {
        return Status::NotImplemented("unsupported types for take operation");
      }
      if (args[1].kind == DatumKind::ARRAY) {
        Datum r;
        RETURN_NOT_OK(CallFunction(ctx, "array_take", opts, {values, args[1]}, &r));
        if (!values_chunked) { *out = r; return Status::OK(); }
        auto c = std::make_shared<ChunkedArray>();
        c->type = r.array->type; c->chunks = {r.array}; c->length = r.array->length;
        *out = Datum(c);
        return Status::OK();
      }
      auto c = std::make_shared<ChunkedArray>();
      c->type = values.type();
      for (auto& chunk : args[1].chunked->chunks) {  // one array_take per index chunk (selection.go:221-234)
        Datum r;
        RETURN_NOT_OK(CallFunction(ctx, "array_take", opts, {values, Datum(chunk)}, &r));
        c->chunks.push_back(r.array);
        c->length += r.array->length;
      }
      *out = Datum(c);
      return Status::OK();
    }), false);
  });
  return reg;
}

namespace {
Status ConcatenateChunks(const ChunkedArray& c, std::shared_ptr<ArrayData>* out) {  // array.Concatenate on device (D2D)
  auto d = std::make_shared<ArrayData>();
  d->type = c.type; d->length = c.length; d->offset = 0;
  const int w = BitWidth(c.type) / 8;
  if (w == 0) return Status::NotImplemented("concatenate of boolean chunks");
  RETURN_NOT_OK(Buffer::Allocate(c.length * w, &d->buffers[1]));
  bool any_nulls = false;
  for (auto& ch : c.chunks) any_nulls = any_nulls || (ch->buffers[0] && ch->null_count != 0);
  if (any_nulls) RETURN_NOT_OK(Buffer::Allocate((c.length + 7) / 8, &d->buffers[0]));
  int64_t pos = 0;
  for (auto& ch : c.chunks) {
    NATIVE(ag_copy_dev(d->buffers[1]->data() + pos * w, ch->buffers[1]->data() + ch->offset * w, (size_t)(ch->length * w), nullptr));
    if (any_nulls) {
      if (ch->buffers[0] && ch->null_count != 0) NATIVE(ag_bitmap_copy_dev(ch->buffers[0]->data(), ch->offset, ch->length, d->buffers[0]->data(), pos, nullptr));
      else NATIVE(ag_bitmap_set_dev(d->buffers[0]->data(), pos, ch->length, 1, nullptr));
    }
    pos += ch->length;
  }
  d->null_count = any_nulls ? kUnknownNullCount : 0;
  *out = d;
  return Status::OK();
}

// dictionaryEncodeAction (kernels/vector_hash.go:144-241) over doAppendNumeric (:359-385): the chunks of a chunked input
// are concatenated on the device and encoded in one call, so every chunk's indices point into one dictionary
// (dictionaryEncodeFinalize :854-872); the output chunks are zero-copy slices of one indices buffer.
Status DictionaryEncodeImpl(const DictionaryEncodeOptions& opts, const Datum& values, Datum* out) {
  if (opts.NullEncoding != NullEncodingMask && opts.NullEncoding != NullEncodingEncode)
    return Status::Invalid("invalid null encoding behavior " + std::to_string((int)opts.NullEncoding));  // :103-104
  if (values.kind != DatumKind::ARRAY && values.kind != DatumKind::CHUNKED) return Status::NotImplemented("dictionary_encode takes an array or a chunked array");
  if (values.type() == Type::DICTIONARY) { *out = values; return Status::OK(); }  // dictionaryEncodeIdentity :473-500
  const Type t = values.type();
  if (!IsNumeric(t)) return Status::NotImplemented(std::string("dictionary_encode: unsupported type ") + TypeName(t));
  const int bw = BitWidth(t);
  std::shared_ptr<ArrayData> a;
  if (values.kind == DatumKind::ARRAY) a = values.array;
  else if (values.chunked->chunks.size() == 1) a = values.chunked->chunks[0];
  else if (values.chunked->chunks.empty()) { a = std::make_shared<ArrayData>(); a->type = t; }
  else RETURN_NOT_OK(ConcatenateChunks(*values.chunked, &a));
  if (a->length >= (1ll << 31)) return Status::NotImplemented("dictionary_encode: more than 2^31-1 rows per call");
  const bool encode = opts.NullEncoding == NullEncodingEncode;
  const bool has_valid = a->buffers[0] && a->null_count != 0;
  const int64_t n = a->length;
  std::shared_ptr<Buffer> idx, idx_valid, dict, dict_valid, counts;
  RETURN_NOT_OK(Buffer::Allocate(std::max<int64_t>(n, 1) * 4, &idx));
  RETURN_NOT_OK(Buffer::Allocate(std::max<int64_t>(n, 1) * (bw / 8), &dict));
  const int64_t bm = ((n + 31) / 32) * 4 + 4;
  if (has_valid && !encode) RETURN_NOT_OK(Buffer::Allocate(bm, &idx_valid));
  if (has_valid && encode) RETURN_NOT_OK(Buffer::Allocate(bm, &dict_valid));
  RETURN_NOT_OK(Buffer::Allocate(16, &counts));
  NATIVE(ag_dictionary_encode_dev(bw, a->buffers[1] ? a->buffers[1]->data() : nullptr, has_valid ? a->buffers[0]->data() : nullptr, a->offset, n,
                                  (int)opts.NullEncoding, (int32_t*)idx->data(), idx_valid ? idx_valid->data() : nullptr, dict->data(),
                                  dict_valid ? dict_valid->data() : nullptr, n, (int64_t*)counts->data(), nullptr));
  int64_t c[2] = {0, 0};
  RETURN_NOT_OK(counts->ToHost(c, 16));
  auto d = std::make_shared<ArrayData>();
  d->type = t; d->length = c[0];
  d->buffers[1] = dict;
  d->buffers[0] = dict_valid;
  d->null_count = !dict_valid ? 0 : (a->null_count > 0 ? 1 : kUnknownNullCount);  // the one null entry, when the input has a null
  auto r = std::make_shared<ArrayData>();
  r->type = Type::DICTIONARY; r->length = n;
  r->buffers[1] = idx;
  r->buffers[0] = idx_valid;
  r->null_count = idx_valid ? c[1] : 0;
  r->dictionary = d;
  if (values.kind == DatumKind::ARRAY) { *out = Datum(r); return Status::OK(); }
  auto res = std::make_shared<ChunkedArray>();
  res->type = Type::DICTIONARY;
  int64_t pos = 0;
  for (auto& ch : values.chunked->chunks) {
    res->chunks.push_back(r->Slice(pos, ch->length));
    pos += ch->length;
  }
  res->length = pos;
  *out = Datum(res);
  return Status::OK();
}
}  // namespace

// arithmetic.go:1090-1142
static Status CumulativeImpl(const ExecCtx& ctx, const char* fn, const CumulativeOptions& opts, const Datum& values, Datum* out) {
  if (values.kind == DatumKind::SCALAR) {  // the vector executor promotes a scalar argument to a length-1 array
    if (!values.scalar) return Status::Invalid("cumulative sum: empty datum");
    std::shared_ptr<ArrayData> one;
    const uint8_t zero = 0;
    RETURN_NOT_OK(ArrayData::FromHost(values.scalar->type, 1, 0, values.scalar->valid ? nullptr : &zero, values.scalar->value,
                                      values.scalar->valid ? 0 : 1, &one));
    return CallFunction(ctx, fn, &opts, {Datum(one)}, out);
  }
  return CallFunction(ctx, fn, &opts, {values}, out);
}
Status CumulativeSum(const ExecCtx& ctx, const CumulativeOptions& opts, const Datum& values, Datum* out) { return CumulativeImpl(ctx, "cumulative_sum", opts, values, out); }
Status CumulativeSumChecked(const ExecCtx& ctx, const CumulativeOptions& opts, const Datum& values, Datum* out) { return CumulativeImpl(ctx, "cumulative_sum_checked", opts, values, out); }

Status CastDatum(const ExecCtx& ctx, const Datum& val, const CastOptions& opts, Datum* out) {  // cast.go:919-921
  return CallFunction(ctx, "cast", &opts, {val}, out);
}

static Status ArithImpl(const ExecCtx& ctx, const ArithmeticOptions& opts, const char* fn, const Datum& l, const Datum& r, Datum* out) {
  std::string name = fn;
  if (opts.NoCheckOverflow) name += "_unchecked";
  return CallFunction(ctx, name, nullptr, {l, r}, out);
}
Status Add(const ExecCtx& ctx, const ArithmeticOptions& o, const Datum& l, const Datum& r, Datum* out) { return ArithImpl(ctx, o, "add", l, r, out); }
Status Subtract(const ExecCtx& ctx, const ArithmeticOptions& o, const Datum& l, const Datum& r, Datum* out) { return ArithImpl(ctx, o, "sub", l, r, out); }
Status Multiply(const ExecCtx& ctx, const ArithmeticOptions& o, const Datum& l, const Datum& r, Datum* out) { return ArithImpl(ctx, o, "multiply", l, r, out); }
// ---- sort_indices / unique / is_in (SURVEY 8f rank 3): single fixed-width column, anything else is ErrNotImplemented
// like the reference's type switches (vector_sort.go:183-185, scalar_set_lookup.go:270-272) ------------------------
static Status OneArray(const Datum& d, const char* fn, std::shared_ptr<ArrayData>* out) {
  if (d.kind == DatumKind::ARRAY) { *out = d.array; return Status::OK(); }
  if (d.kind == DatumKind::CHUNKED && d.chunked->chunks.size() == 1) { *out = d.chunked->chunks[0]; return Status::OK(); }
  return Status::NotImplemented(std::string(fn) + ": the GPU kernel takes one array (a multi-chunk input is merged by the parent registry's function)");
}
static Status MakeOut(Type t, int64_t len, std::shared_ptr<Buffer> data, std::shared_ptr<Buffer> valid, int64_t nulls, Datum* out) {
  auto a = std::make_shared<ArrayData>();
  a->type = t; a->length = len; a->offset = 0; a->null_count = nulls;
  a->buffers[0] = valid; a->buffers[1] = data;
  *out = Datum(a);
  return Status::OK();
}

Status SortIndices(const ExecCtx& ctx, const Datum& input, const SortOptions& opts, Datum* out) {
  std::shared_ptr<ArrayData> a;
  RETURN_NOT_OK(OneArray(input, "sort_indices", &a));
  if (!IsInteger(a->type) && !IsFloating(a->type)) return Status::NotImplemented(std::string("unsupported type for sort_indices operation: ") + TypeName(a->type));
  std::shared_ptr<Buffer> idx;
  RETURN_NOT_OK(Buffer::Allocate(std::max<int64_t>(a->length, 1) * 8, &idx));
  int64_t nulls = 0, nans = 0;
  const uint8_t* valid = (a->buffers[0] && a->null_count != 0) ? a->buffers[0]->data() : nullptr;
  NATIVE(ag_sort_indices_dev((int)a->type, a->buffers[1] ? a->buffers[1]->data() : nullptr, valid, a->offset, a->length, (int)opts.Order, (int)opts.Placement,
                             (uint64_t*)idx->data(), &nulls, &nans, nullptr));
  return MakeOut(Type::UINT64, a->length, idx, nullptr, 0, out);
}

Status Unique(const ExecCtx& ctx, const Datum& values, Datum* out) {
  std::shared_ptr<ArrayData> a;
  RETURN_NOT_OK(OneArray(values, "unique", &a));
  const int bw = BitWidth(a->type);
  if (bw != 8 && bw != 16 && bw != 32 && bw != 64) return Status::NotImplemented(std::string("unique: unsupported type ") + TypeName(a->type));
  const bool has_valid = a->buffers[0] && a->null_count != 0;
  std::shared_ptr<Buffer> data, valid, len;
  RETURN_NOT_OK(Buffer::Allocate(std::max<int64_t>(a->length, 1) * (bw / 8), &data));
  if (has_valid) RETURN_NOT_OK(Buffer::Allocate(((a->length + 31) / 32) * 4 + 4, &valid));
  RETURN_NOT_OK(Buffer::Allocate(16, &len));
  NATIVE(ag_unique_dev(bw, a->buffers[1] ? a->buffers[1]->data() : nullptr, has_valid ? a->buffers[0]->data() : nullptr, a->offset, a->length, data->data(),
                       has_valid ? valid->data() : nullptr, a->length, (int64_t*)len->data(), nullptr));
  int64_t k = 0;
  RETURN_NOT_OK(len->ToHost(&k, 8));
  return MakeOut(a->type, k, data, valid, has_valid ? kUnknownNullCount : 0, out);
}

Status IsIn(const ExecCtx& ctx, const SetLookupOptions& opts, const Datum& values, Datum* out) {
  std::shared_ptr<ArrayData> a;
  RETURN_NOT_OK(OneArray(values, "is_in", &a));
  if (!opts.ValueSet) return Status::Invalid("is_in: SetLookupOptions.ValueSet is required");
  if (opts.ValueSet->type != a->type) return Status::NotImplemented("is_in: the value set must have the input's type (casts are left to the parent registry)");
  const int bw = BitWidth(a->type);
  if (bw != 8 && bw != 16 && bw != 32 && bw != 64) return Status::Invalid(std::string("unsupported type ") + TypeName(a->type) + " for is_in function");
  const ArrayData& s = *opts.ValueSet;
  std::shared_ptr<Buffer> data, valid, cnt;
  const int64_t bm = ((a->length + 31) / 32) * 4 + 4;
  RETURN_NOT_OK(Buffer::Allocate(bm, &data));
  RETURN_NOT_OK(Buffer::Allocate(bm, &valid));
  RETURN_NOT_OK(Buffer::Allocate(8, &cnt));
  NATIVE(ag_is_in_dev(bw, a->buffers[1] ? a->buffers[1]->data() : nullptr, (a->buffers[0] && a->null_count != 0) ? a->buffers[0]->data() : nullptr, a->offset, a->length,
                      s.buffers[1] ? s.buffers[1]->data() : nullptr, (s.buffers[0] && s.null_count != 0) ? s.buffers[0]->data() : nullptr, s.offset, s.length,
                      (int)opts.NullBehavior, data->data(), valid->data(), (int64_t*)cnt->data(), nullptr));
  int64_t nulls = 0;
  RETURN_NOT_OK(cnt->ToHost(&nulls, 8));
  return MakeOut(Type::BOOL, a->length, data, nulls ? valid : nullptr, nulls, out);
}

Status DictionaryEncode(const ExecCtx& ctx, const DictionaryEncodeOptions& opts, const Datum& values, Datum* out) {
  return CallFunction(ctx, "dictionary_encode", &opts, {values}, out);
}

Status Filter(const ExecCtx& ctx, const Datum& values, const Datum& filter, const FilterOptions& opts, Datum* out) {
  return CallFunction(ctx, "filter", &opts, {values, filter}, out);
}
Status Take(const ExecCtx& ctx, const TakeOptions& opts, const Datum& values, const Datum& indices, Datum* out) {
  return CallFunction(ctx, "take", &opts, {values, indices}, out);
}

}  // namespace compute

// ======================================================================================
// math
// ======================================================================================
namespace math {
template <typename T, typename F>
static Status SumImpl(const ArrayData& a, Type want, T* out, F&& fn) {
  if (a.type != want) return Status::TypeError(std::string("Sum: expected ") + TypeName(want) + " got " + TypeName(a.type));
  *out = T(0);
  if (a.length == 0) return Status::OK();  // float64.go:35-37
  std::shared_ptr<Buffer> res;
  RETURN_NOT_OK(Buffer::Allocate(8, &res));
  NATIVE(fn((const T*)(a.buffers[1]->data()) + a.offset, (size_t)a.length, (T*)res->data(), nullptr));
  return res->ToHost(out, 8);
}
Status SumFloat64(const ArrayData& a, double* out) { return SumImpl<double>(a, Type::FLOAT64, out, ag_sum_f64_dev); }
Status SumInt64(const ArrayData& a, int64_t* out) { return SumImpl<int64_t>(a, Type::INT64, out, ag_sum_i64_dev); }
Status SumUint64(const ArrayData& a, uint64_t* out) { return SumImpl<uint64_t>(a, Type::UINT64, out, ag_sum_u64_dev); }
Status SumFloat64ReferenceOrder(const ArrayData& a, double* out) { return SumImpl<double>(a, Type::FLOAT64, out, ag_sum_f64_reforder_dev); }
}  // namespace math

}  // namespace arrowgpu
