// capi.cc — flat C surface over the C++ host mirror so that tests (ctypes) can drive
// CallFunction / Add / Filter / Take / Sum exactly like the reference's Go tests do.
// Not part of the drop-in boundary (that is include/arrowgpu.h); this is the harness's door
// into the host layer because no Go toolchain exists here.
#include "arrowgpu_compute.h"

#include <string.h>
#include <string>

using namespace arrowgpu;
using namespace arrowgpu::compute;

static thread_local std::string g_err;
static int fail(const Status& s) { g_err = s.msg; return s.code; }
#define AGX_TRY(expr) do { Status _s = (expr); if (!_s.ok()) return fail(_s); } while (0)

extern "C" {

typedef struct agx_datum { Datum d; } agx_datum;

const char* agx_last_error(void) { return g_err.c_str(); }

int agx_array_from_host(int type, int64_t length, int64_t offset, const uint8_t* validity, const void* values,
                        int64_t null_count, agx_datum** out) {
  std::shared_ptr<ArrayData> a;
  AGX_TRY(ArrayData::FromHost((Type)type, length, offset, validity, values, null_count, &a));
  *out = new agx_datum{Datum(a)};
  return AG_OK;
}
int agx_scalar(int type, int valid, const void* value, agx_datum** out) {
  auto s = std::make_shared<Scalar>();
  s->type = (Type)type; s->valid = valid != 0;
  if (value) memcpy(s->value, value, (size_t)((BitWidth((Type)type) + 7) / 8));
  *out = new agx_datum{Datum(s)};
  return AG_OK;
}
int agx_chunked(int type, agx_datum** chunks, int n, agx_datum** out) {
  auto c = std::make_shared<ChunkedArray>();
  c->type = (Type)type;
  for (int i = 0; i < n; ++i) {
    if (chunks[i]->d.kind != DatumKind::ARRAY || chunks[i]->d.array->type != c->type) return fail(Status::Invalid("chunked: chunks must be arrays of the chunked type"));
    c->chunks.push_back(chunks[i]->d.array);
    c->length += chunks[i]->d.array->length;
  }
  *out = new agx_datum{Datum(c)};
  return AG_OK;
}
int agx_slice(agx_datum* a, int64_t off, int64_t len, agx_datum** out) {
  if (a->d.kind != DatumKind::ARRAY) return fail(Status::Invalid("slice: not an array"));
  if (off < 0 || len < 0 || off + len > a->d.array->length) return fail(Status::Invalid("slice: out of range"));
  *out = new agx_datum{Datum(a->d.array->Slice(off, len))};
  return AG_OK;
}
void agx_release(agx_datum* d) { delete d; }
int agx_kind(agx_datum* d) { return (int)d->d.kind; }
int agx_type(agx_datum* d) { return (int)d->d.type(); }
int64_t agx_len(agx_datum* d) { return d->d.Len(); }
int64_t agx_offset(agx_datum* d) { return d->d.kind == DatumKind::ARRAY ? d->d.array->offset : 0; }
int agx_has_validity(agx_datum* d) { return d->d.kind == DatumKind::ARRAY && d->d.array->buffers[0] != nullptr; }
int64_t agx_null_count_raw(agx_datum* d) { return d->d.kind == DatumKind::ARRAY ? d->d.array->null_count : 0; }
int agx_num_chunks(agx_datum* d) { return d->d.kind == DatumKind::CHUNKED ? (int)d->d.chunked->chunks.size() : 0; }
int agx_chunk(agx_datum* d, int i, agx_datum** out) {
  if (d->d.kind != DatumKind::CHUNKED || i < 0 || i >= (int)d->d.chunked->chunks.size()) return fail(Status::Invalid("chunk: out of range"));
  *out = new agx_datum{Datum(d->d.chunked->chunks[i])};
  return AG_OK;
}
int agx_array_to_host(agx_datum* d, void* values, uint8_t* validity, int64_t* null_count) {
  if (d->d.kind != DatumKind::ARRAY) return fail(Status::Invalid("to_host: not an array"));
  AGX_TRY(d->d.array->ToHost(values, validity, null_count));
  return AG_OK;
}

// opt_kind: 0 none, 1 ArithmeticOptions{NoCheckOverflow=opt_value}, 2 FilterOptions{NullSelection=opt_value},
//           3 TakeOptions{BoundsCheck=opt_value}
int agx_call_function(const char* name, int opt_kind, int opt_value, agx_datum** args, int nargs, agx_datum** out) {
  std::vector<Datum> a;
  for (int i = 0; i < nargs; ++i) a.push_back(args[i]->d);
  ArithmeticOptions ao; FilterOptions fo; TakeOptions to;
  const FunctionOptions* opts = nullptr;
  if (opt_kind == 1) { ao.NoCheckOverflow = opt_value != 0; opts = &ao; }
  if (opt_kind == 2) { fo.NullSelection = (NullSelectionBehavior)opt_value; opts = &fo; }
  if (opt_kind == 3) { to.BoundsCheck = opt_value != 0; opts = &to; }
  ExecCtx ctx;
  Datum r;
  AGX_TRY(CallFunction(ctx, name, opts, a, &r));
  *out = new agx_datum{r};
  return AG_OK;
}
// compute.Add / Subtract / Multiply with ArithmeticOptions (arithmetic.go:1104-1142)
int agx_arith(int which, int no_check_overflow, agx_datum* l, agx_datum* r, agx_datum** out) {
  ArithmeticOptions o; o.NoCheckOverflow = no_check_overflow != 0;
  ExecCtx ctx; Datum res;
  Status s = which == 0 ? Add(ctx, o, l->d, r->d, &res) : (which == 1 ? Subtract(ctx, o, l->d, r->d, &res) : Multiply(ctx, o, l->d, r->d, &res));
  if (!s.ok()) return fail(s);
  *out = new agx_datum{res};
  return AG_OK;
}
// compute.CumulativeSum / CumulativeSumChecked with CumulativeOptions{Start, SkipNulls}; start may be NULL
int agx_cumulative_sum(agx_datum* d, int checked, int skip_nulls, agx_datum* start, agx_datum** out) {
  CumulativeOptions o; o.SkipNulls = skip_nulls != 0;
  if (start) { if (start->d.kind != DatumKind::SCALAR) return fail(Status::Invalid("start must be a scalar")); o.Start = start->d.scalar; }
  ExecCtx ctx; Datum res;
  AGX_TRY(checked ? CumulativeSumChecked(ctx, o, d->d, &res) : CumulativeSum(ctx, o, d->d, &res));
  *out = new agx_datum{res};
  return AG_OK;
}
// compute.CastDatum with CastOptions{ToType, AllowIntOverflow, AllowFloatTruncate} (cast.go:919-921)
int agx_cast(agx_datum* d, int to_type, int allow_int_overflow, int allow_float_truncate, agx_datum** out) {
  CastOptions o; o.ToType = (Type)to_type; o.AllowIntOverflow = allow_int_overflow != 0; o.AllowFloatTruncate = allow_float_truncate != 0;
  ExecCtx ctx; Datum res;
  AGX_TRY(CastDatum(ctx, d->d, o, &res));
  *out = new agx_datum{res};
  return AG_OK;
}
// compute.SortIndices(SortOptions{Order, NullPlacement}) / compute.Unique / compute.IsIn(SetLookupOptions{ValueSet, NullBehavior})
int agx_sort_indices(agx_datum* d, int order, int null_placement, agx_datum** out) {
  SortOptions o; o.Order = (SortOrder)order; o.Placement = (NullPlacement)null_placement;
  ExecCtx ctx; Datum res;
  AGX_TRY(CallFunction(ctx, "sort_indices", &o, {d->d}, &res));
  *out = new agx_datum{res};
  return AG_OK;
}
int agx_unique(agx_datum* d, agx_datum** out) {
  ExecCtx ctx; Datum res;
  AGX_TRY(CallFunction(ctx, "unique", nullptr, {d->d}, &res));
  *out = new agx_datum{res};
  return AG_OK;
}
int agx_is_in(agx_datum* d, agx_datum* value_set, int null_behavior, agx_datum** out) {
  if (value_set->d.kind != DatumKind::ARRAY) return fail(Status::Invalid("is_in: the value set must be an array"));
  SetLookupOptions o; o.ValueSet = value_set->d.array; o.NullBehavior = (NullMatchingBehavior)null_behavior;
  ExecCtx ctx; Datum res;
  AGX_TRY(CallFunction(ctx, "is_in", &o, {d->d}, &res));
  *out = new agx_datum{res};
  return AG_OK;
}
// compute.DictionaryEncode(DictionaryEncodeOptions{NullEncoding}); agx_dictionary: the dictionary of a dictionary array
int agx_dictionary_encode(agx_datum* d, int null_encoding, agx_datum** out) {
  DictionaryEncodeOptions o; o.NullEncoding = (NullEncodingBehavior)null_encoding;
  ExecCtx ctx; Datum res;
  AGX_TRY(DictionaryEncode(ctx, o, d->d, &res));
  *out = new agx_datum{res};
  return AG_OK;
}
int agx_dictionary(agx_datum* d, agx_datum** out) {
  if (d->d.kind != DatumKind::ARRAY || !d->d.array->dictionary) return fail(Status::Invalid("dictionary: not a dictionary array"));
  *out = new agx_datum{Datum(d->d.array->dictionary)};
  return AG_OK;
}
int agx_scalar_value(agx_datum* d, int* valid, void* value8) {
  if (d->d.kind != DatumKind::SCALAR) return fail(Status::Invalid("scalar_value: not a scalar"));
  *valid = d->d.scalar->valid ? 1 : 0;
  memcpy(value8, d->d.scalar->value, 8);
  return AG_OK;
}
int agx_sum_f64(agx_datum* d, int reference_order, double* out) {
  if (d->d.kind != DatumKind::ARRAY) return fail(Status::Invalid("sum: not an array"));
  AGX_TRY(reference_order ? math::SumFloat64ReferenceOrder(*d->d.array, out) : math::SumFloat64(*d->d.array, out));
  return AG_OK;
}
int agx_sum_i64(agx_datum* d, int64_t* out) {
  if (d->d.kind != DatumKind::ARRAY) return fail(Status::Invalid("sum: not an array"));
  AGX_TRY(math::SumInt64(*d->d.array, out));
  return AG_OK;
}
int agx_sum_u64(agx_datum* d, uint64_t* out) {
  if (d->d.kind != DatumKind::ARRAY) return fail(Status::Invalid("sum: not an array"));
  AGX_TRY(math::SumUint64(*d->d.array, out));
  return AG_OK;
}

// Arrow C Device Data Interface: export an Array datum / import one (takes ownership of *in)
int agx_export_device(agx_datum* d, struct ArrowDeviceArray* out, struct ArrowSchema* out_schema) {
  if (d->d.kind != DatumKind::ARRAY) return fail(Status::Invalid("export: not an array"));
  AGX_TRY(d->d.array->ExportDevice(out, out_schema));
  return AG_OK;
}
int agx_import_device(struct ArrowDeviceArray* in, const struct ArrowSchema* schema, agx_datum** out) {
  std::shared_ptr<ArrayData> a;
  AGX_TRY(ArrayData::ImportDevice(in, schema, &a));
  *out = new agx_datum{Datum(a)};
  return AG_OK;
}

// metadata-only pieces (run without a GPU)
int agx_iterate_spans(const int64_t* lens_flat, const int* nchunks, const int* is_chunked, int nargs, int64_t max_chunk,
                      int64_t* out_pos_len, int* out_chunk_idx, int cap, int* n_out) {
  std::vector<std::vector<int64_t>> lens(nargs);
  std::vector<bool> chunked(nargs);
  int k = 0;
  for (int i = 0; i < nargs; ++i) {
    chunked[i] = is_chunked[i] != 0;
    for (int j = 0; j < nchunks[i]; ++j) lens[i].push_back(lens_flat[k++]);
  }
  std::vector<SpanPiece> pieces;
  AGX_TRY(IterateExecSpans(lens, chunked, max_chunk, &pieces));
  *n_out = (int)pieces.size();
  for (int p = 0; p < (int)pieces.size() && p < cap; ++p) {
    out_pos_len[2 * p] = pieces[p].pos;
    out_pos_len[2 * p + 1] = pieces[p].len;
    for (int i = 0; i < nargs; ++i) out_chunk_idx[p * nargs + i] = pieces[p].chunk_index[i];
  }
  return AG_OK;
}
int agx_function_names(char* buf, int64_t buflen) {
  std::string all;
  for (auto& n : GetFunctionRegistry()->GetFunctionNames()) all += n + "\n";
  if ((int64_t)all.size() + 1 > buflen) return fail(Status::Invalid("buffer too small"));
  memcpy(buf, all.c_str(), all.size() + 1);
  return AG_OK;
}
int agx_common_numeric(const int* types, int n) {  // commonNumeric, utils.go:178-240 (0 = none)
  std::vector<Type> t;
  for (int i = 0; i < n; ++i) t.push_back((Type)types[i]);
  return (int)CommonNumeric(t);
}
// DispatchBest: rewrites `types` to the signature the call would run with (after implicit promotion)
int agx_dispatch_best(const char* name, int* types, int n) {
  const Function* f = GetFunctionRegistry()->GetFunction(name);
  if (!f) return fail(Status::Make(AG_ERR_INVALID, std::string("no function registered with name: ") + name));
  if (f->Kind() != FuncKind::SCALAR) return fail(Status::Invalid("dispatch_best: scalar functions only"));
  std::vector<Type> t;
  for (int i = 0; i < n; ++i) t.push_back((Type)types[i]);
  const exec::ScalarKernel* k;
  AGX_TRY(static_cast<const ScalarFunction*>(f)->DispatchBest(&t, &k));
  for (int i = 0; i < n; ++i) types[i] = (int)t[i];
  return AG_OK;
}
// dispatch-only check: does `name` have a kernel for these input types?  (no device work)
int agx_dispatch(const char* name, const int* types, int n) {
  const Function* f = GetFunctionRegistry()->GetFunction(name);
  if (!f) return fail(Status::Make(AG_ERR_INVALID, std::string("no function registered with name: ") + name));
  std::vector<Type> t;
  for (int i = 0; i < n; ++i) t.push_back((Type)types[i]);
  if (f->Kind() == FuncKind::SCALAR) { const exec::ScalarKernel* k; AGX_TRY(static_cast<const ScalarFunction*>(f)->DispatchExact(t, &k)); }
  else if (f->Kind() == FuncKind::VECTOR) { const exec::VectorKernel* k; AGX_TRY(static_cast<const VectorFunction*>(f)->DispatchExact(t, &k)); }
  return AG_OK;
}

// ---- ipc: file reader + device streams -------------------------------------------------------------------------
typedef struct agx_ipc_reader { std::shared_ptr<ipc::FileReader> r; } agx_ipc_reader;

int agx_ipc_open(const uint8_t* data, int64_t size, agx_ipc_reader** out) {
  std::unique_ptr<ipc::FileReader> r;
  AGX_TRY(ipc::FileReader::Open(data, size, &r));
  *out = new agx_ipc_reader{std::shared_ptr<ipc::FileReader>(std::move(r))};
  return AG_OK;
}
void agx_ipc_close(agx_ipc_reader* h) { delete h; }
int agx_ipc_num_fields(agx_ipc_reader* h) { return (int)h->r->schema().size(); }
int agx_ipc_num_records(agx_ipc_reader* h) { return h->r->NumRecords(); }
int agx_ipc_version(agx_ipc_reader* h) { return h->r->version(); }
int agx_ipc_field(agx_ipc_reader* h, int i, char* name, int64_t cap, int* type, int* nullable) {
  if (i < 0 || i >= (int)h->r->schema().size()) return fail(Status::Invalid("ipc: field index out of range"));
  const ipc::Field& f = h->r->schema()[(size_t)i];
  if ((int64_t)f.name.size() + 1 > cap) return fail(Status::Invalid("ipc: name buffer too small"));
  memcpy(name, f.name.c_str(), f.name.size() + 1);
  *type = (int)f.type;
  *nullable = f.nullable ? 1 : 0;
  return AG_OK;
}
// cols: 6 int64 per field {length, null_count, validity_offset, validity_length, data_offset, data_length}
int agx_ipc_layout(agx_ipc_reader* h, int i, int64_t* rows, int64_t* body_offset, int64_t* body_length, int64_t* cols) {
  std::vector<ipc::ColumnLayout> L;
  AGX_TRY(h->r->Layout(i, rows, body_offset, body_length, &L));
  for (size_t c = 0; c < L.size(); ++c) {
    int64_t* o = cols + 6 * c;
    o[0] = L[c].length; o[1] = L[c].null_count; o[2] = L[c].validity_offset; o[3] = L[c].validity_length; o[4] = L[c].data_offset; o[5] = L[c].data_length;
  }
  return AG_OK;
}
int agx_ipc_read_batch(agx_ipc_reader* h, int i, int64_t* rows, agx_datum** cols) {
  ipc::RecordBatch rb;
  AGX_TRY(h->r->RecordBatchAt(i, &rb));
  *rows = rb.num_rows;
  for (size_t c = 0; c < rb.columns.size(); ++c) cols[c] = new agx_datum{Datum(rb.columns[c])};
  return AG_OK;
}
int agx_ipc_export_stream(agx_ipc_reader* h, struct ArrowDeviceArrayStream* out) {
  AGX_TRY(ipc::ExportDeviceStream(h->r, out));
  return AG_OK;
}
// Drains `stream`; batches come back column-major: cols[b * nfields + c].  *nbatches in: capacity, out: count.
int agx_ipc_import_stream(struct ArrowDeviceArrayStream* stream, int* nfields, int* types, int max_fields,
                          int* nbatches, int64_t* rows, agx_datum** cols) {
  std::vector<ipc::Field> schema;
  std::vector<ipc::RecordBatch> batches;
  AGX_TRY(ipc::ImportDeviceStream(stream, &schema, &batches));
  if ((int)schema.size() > max_fields || (int)batches.size() > *nbatches) return fail(Status::Invalid("ipc: output arrays too small"));
  *nfields = (int)schema.size();
  for (size_t c = 0; c < schema.size(); ++c) types[c] = (int)schema[c].type;
  *nbatches = (int)batches.size();
  for (size_t b = 0; b < batches.size(); ++b) {
    rows[b] = batches[b].num_rows;
    for (size_t c = 0; c < schema.size(); ++c) cols[b * schema.size() + c] = new agx_datum{Datum(batches[b].columns[c])};
  }
  return AG_OK;
}

}  // extern "C"
