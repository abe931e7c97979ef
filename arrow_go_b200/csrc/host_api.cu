// host_api.cu — the HOST-pointer flavour of every compute entry point.
//
// This is the form a per-span exec.ArrayKernelExec binds through cgo: it receives the raw
// bytes of ArraySpan.Buffers[i].Buf exactly like the reference's asm stubs do
// (arrow/compute/internal/kernels/base_arithmetic_avx2_amd64.go:35-39) and returns when the
// output bytes are in host memory.  Each call owns pooled streams for its duration, stages its
// operands into stream-ordered device temporaries and runs the SAME kernels as the *_dev
// flavour (so results are bit-identical between the two).
//
// Elementwise arithmetic and comparisons are pipelined in row chunks over three streams so
// that H2D of chunk k+1, the kernel of chunk k and D2H of chunk k-1 overlap (PCIe is full
// duplex; the kernels are ~100x faster than the link).  Buffers obtained from ag_host_alloc /
// ag_host_register are DMA'd directly; pageable memory still works but the driver bounces it
// through its own pinned staging area.
#include "common.cuh"

#include <stdlib.h>
#include <string.h>
#include <vector>

namespace ag {

// forward declarations of the device-flavour implementations
ag_status arith_binary_dev(int type, int8_t op, int shape, const void* l, const void* r, void* out, int64_t n, cudaStream_t st);
ag_status arith_unary_same_dev(int type, int8_t op, const void* in, void* out, int64_t n, cudaStream_t st);
ag_status arith_unary_diff_dev(int itype, int otype, int8_t op, const void* in, void* out, int64_t n, cudaStream_t st);
ag_status arith_checked_dev(int type, int8_t op, int shape, const void* l, const uint8_t* lvalid, int64_t loff,
                            const void* r, const uint8_t* rvalid, int64_t roff, void* out, int64_t n, int64_t* d_first_bad, cudaStream_t st);
ag_status error_word_reset(int64_t* d_word, cudaStream_t st);
ag_status arith_unary_checked_dev(int type, int8_t op, const void* in, void* out, int64_t n, int64_t* d_first_bad, cudaStream_t st);
ag_status cast_numeric_dev(int itype, int otype, const void* in, const uint8_t* valid, int64_t voff, void* out, int64_t n,
                           int allow_int_overflow, int allow_float_truncate, int64_t* first_bad, int64_t row_base, cudaStream_t st);
ag_status cumulative_sum_dev(int type, const void* in, const uint8_t* valid, int64_t voff, int64_t n, int skip_nulls, int checked,
                             void* out, uint8_t* out_valid, int64_t ooff, void* d_state, int64_t* d_first_bad, cudaStream_t st);
ag_status cumulative_sum_state_init(void* d_state, int type, const void* start_host, cudaStream_t st);
ag_status compare_dev(int type, int cmp, int shape, const void* l, const void* r, uint8_t* out, int64_t n, int off, cudaStream_t st);
ag_status bitmap_op_dev(int bitop, const uint8_t* l, int64_t loff, const uint8_t* r, int64_t roff, uint8_t* out, int64_t ooff, int64_t n, cudaStream_t st);
ag_status bitmap_copy_dev(const uint8_t* src, int64_t soff, int64_t n, uint8_t* dst, int64_t doff, bool invert, cudaStream_t st);
ag_status bitmap_set_dev(uint8_t* bits, int64_t off, int64_t n, int value, cudaStream_t st);
ag_status bitmap_popcount_dev(const uint8_t* bits, int64_t off, int64_t n, int64_t* d_count, cudaStream_t st);
ag_status kleene_dev(int kop, const uint8_t* lvalid, const uint8_t* ldata, int64_t loff, const uint8_t* rvalid, const uint8_t* rdata,
                     int64_t roff, uint8_t* out_valid, uint8_t* out_data, int64_t ooff, int64_t n, cudaStream_t st);
ag_status filter_output_size_dev(const uint8_t* mask, const uint8_t* mvalid, int64_t moff, int64_t n, int null_selection, int64_t* d_out_len, cudaStream_t st);
ag_status filter_primitive_dev(int bit_width, const void* vals, const uint8_t* vvalid, int64_t voff, const uint8_t* mask, const uint8_t* mvalid,
                               int64_t moff, int64_t n, int null_selection, void* out, uint8_t* out_valid, int64_t capacity, int64_t* d_out_len, cudaStream_t st);
ag_status take_indices_dev(int index_width, const uint8_t* mask, const uint8_t* mvalid, int64_t moff, int64_t n, int null_selection,
                           void* out_idx, uint8_t* out_valid, int64_t capacity, int64_t* d_out_len, cudaStream_t st);
ag_status is_in_dev(int bit_width, const void* vals, const uint8_t* valid, int64_t off, int64_t n, const void* set, const uint8_t* set_valid,
                    int64_t set_off, int64_t set_n, int null_behavior, uint8_t* out_data, uint8_t* out_valid, int64_t* d_null_count, cudaStream_t st);
ag_status unique_dev(int bit_width, const void* vals, const uint8_t* valid, int64_t off, int64_t n, void* out, uint8_t* out_valid, int64_t capacity,
                     int64_t* d_out_len, cudaStream_t st);
ag_status dictionary_encode_dev(int bit_width, const void* vals, const uint8_t* valid, int64_t off, int64_t n, int null_encoding, int32_t* indices,
                                uint8_t* indices_valid, void* dict, uint8_t* dict_valid, int64_t dict_capacity, int64_t* d_counts, cudaStream_t st);
ag_status sort_indices_dev(int type, const void* vals, const uint8_t* valid, int64_t voff, int64_t n, int order, int null_placement,
                           uint64_t* d_out, int64_t* nulls_out, int64_t* nans_out, cudaStream_t st);
ag_status take_primitive_dev(int bit_width, const void* vals, const uint8_t* vvalid, int64_t voff, int64_t vlen, int idx_width, int idx_signed,
                             const void* idx, const uint8_t* ivalid, int64_t ioff, int64_t n, int bounds_check, void* out, uint8_t* out_valid,
                             int64_t* d_bad_pos, cudaStream_t st);

// Stream-ordered temporaries of one host call; freed (async) when the call returns.
struct Temps {
  cudaStream_t st;
  std::vector<void*> ptrs;
  explicit Temps(cudaStream_t s) : st(s) {}
  ag_status alloc(void** p, size_t nbytes) {
    AG_TRY(dev_alloc_async(p, nbytes + 64, st));  // +64: kernels may read/write whole aligned words at the edges
    ptrs.push_back(*p);
    return AG_OK;
  }
  template <typename T> ag_status alloc_t(T** p, size_t nbytes) { return alloc(reinterpret_cast<void**>(p), nbytes); }
  ~Temps() {
    // An early (error) return may leave H2D / D2H copies of CALLER memory in flight on this pooled stream: wait for
    // them before the function returns and before the stream goes back to the pool.  On the success paths the
    // stream is already idle and this costs a few microseconds.
    cudaStreamSynchronize(st);
    for (void* p : ptrs) cudaFreeAsync(p, st);
  }
};

static inline ag_status h2d(void* d, const void* h, size_t nbytes, cudaStream_t st) {
  if (nbytes) AG_CUDA_TRY(cudaMemcpyAsync(d, h, nbytes, cudaMemcpyHostToDevice, st));
  return AG_OK;
}
static inline ag_status d2h(void* h, const void* d, size_t nbytes, cudaStream_t st) {
  if (nbytes) AG_CUDA_TRY(cudaMemcpyAsync(h, d, nbytes, cudaMemcpyDeviceToHost, st));
  return AG_OK;
}
static inline ag_status sync(cudaStream_t st) { AG_CUDA_TRY(cudaStreamSynchronize(st)); return AG_OK; }

// Upload the bytes of a bitmap range [off, off+n) to a device temp; the device copy keeps the
// same bit phase (off % 8) so kernels address it with bit offset (off & 7).
static ag_status upload_bitmap(Temps& t, const uint8_t* h, int64_t off, int64_t n, uint8_t** d, int64_t* doff) {
  *d = nullptr; *doff = 0;
  if (!h) return AG_OK;
  const int64_t b0 = off >> 3, b1 = (off + n + 7) >> 3;
  AG_TRY(t.alloc_t(d, (size_t)(b1 - b0)));
  AG_TRY(h2d(*d, h + b0, (size_t)(b1 - b0), t.st));
  *doff = off & 7;
  return AG_OK;
}

constexpr int kPipe = 3;
constexpr int64_t kChunkBytes = (int64_t)32 << 20;  // per operand per pipeline stage

struct Pipe {
  CallStream s[kPipe];
  ag_status acquire() { for (auto& c : s) AG_TRY(c.acquire()); return AG_OK; }
  ag_status sync_all() { for (auto& c : s) AG_CUDA_TRY(cudaStreamSynchronize(c.st)); return AG_OK; }
};

// chunked, 3-deep pipelined elementwise call.  in[k] == nullptr marks an operand that is not an array.
template <typename Launch>
static ag_status pipelined_rows(int64_t n, int n_in, const void* const* in, const int* in_width,
                                void* out, int out_width, Launch&& launch) {
  AG_TRY(ensure_init());
  if (n == 0) return AG_OK;
  Pipe pipe;
  AG_TRY(pipe.acquire());
  int wmax = out_width;
  for (int k = 0; k < n_in; ++k) if (in[k] && in_width[k] > wmax) wmax = in_width[k];
  int64_t chunk = kChunkBytes / wmax;
  chunk &= ~(int64_t)1023;
  if (chunk > n) chunk = n;
  const int slots = (n + chunk - 1) / chunk < kPipe ? (int)((n + chunk - 1) / chunk) : kPipe;
  void* d_in[kPipe][4] = {};
  void* d_out[kPipe] = {};
  ag_status rc = AG_OK;
  for (int sl = 0; sl < slots && rc == AG_OK; ++sl) {
    for (int k = 0; k < n_in && rc == AG_OK; ++k)
      if (in[k]) rc = dev_alloc_async(&d_in[sl][k], (size_t)chunk * in_width[k] + 64, pipe.s[sl]);
    if (rc == AG_OK) rc = dev_alloc_async(&d_out[sl], (size_t)chunk * out_width + 64, pipe.s[sl]);
  }
  int64_t ci = 0;
  for (int64_t r0 = 0; r0 < n && rc == AG_OK; r0 += chunk, ++ci) {
    const int sl = (int)(ci % kPipe);
    const int64_t len = (n - r0 < chunk) ? (n - r0) : chunk;
    cudaStream_t st = pipe.s[sl];
    for (int k = 0; k < n_in && rc == AG_OK; ++k)
      if (in[k]) rc = h2d(d_in[sl][k], (const char*)in[k] + r0 * in_width[k], (size_t)len * in_width[k], st);
    if (rc == AG_OK) rc = launch(d_in[sl], d_out[sl], len, st);
    if (rc == AG_OK) rc = d2h((char*)out + r0 * out_width, d_out[sl], (size_t)len * out_width, st);
  }
  for (int sl = 0; sl < slots; ++sl) {
    for (int k = 0; k < n_in; ++k) if (d_in[sl][k]) cudaFreeAsync(d_in[sl][k], pipe.s[sl]);
    if (d_out[sl]) cudaFreeAsync(d_out[sl], pipe.s[sl]);
  }
  ag_status rs = pipe.sync_all();
  return rc != AG_OK ? rc : rs;
}

// Host flavour of the batched-span call.  Spans are cut into pieces of at most one stage (32 MB per operand), pieces
// that continue each other in host memory on every operand are merged (slices of one allocation: a chunked array built
// from NewSlice views), and pieces are PACKED into stages of up to 32 MB: each piece is copied to the next 16-byte
// aligned offset of the stage's device buffers, ONE kernel runs over the packed range (the few padding rows between
// pieces compute garbage nobody reads), and each piece is copied back from the same offset.  So a chunked call with
// 8 MB chunks runs the same 3-deep H2D / kernel / D2H pipeline, with the same stage size, as one contiguous column
// (measured on 100M float64 rows in 200 spans: 38.4 ms per call with one stage per span, 32 ms packed = the contiguous
// call; scripts/e2e_probe.py).
static ag_status host_arith_binary_spans(int type, int8_t op, int shape, const ag_span3* spans, int64_t n_spans) {
  AG_TRY(ensure_init());
  const int w = type_width(type);
  if (w == 0) AG_FAIL(AG_ERR_TYPE, "arith: unsupported type id %d", type);
  if (n_spans < 0 || (n_spans > 0 && !spans)) AG_FAIL(AG_ERR_INVALID, "arith_spans: bad span table");
  const bool la = shape != AG_SHAPE_SA, ra = shape != AG_SHAPE_AS;
  const int64_t chunk = (kChunkBytes / w) & ~(int64_t)1023;   // rows per stage
  const int64_t pad = 16 / w;                                   // pieces start on 16-byte boundaries of the stage
  struct Piece { const char* l; const char* r; char* out; int64_t n; };
  std::vector<Piece> pieces;
  const void* scalar_l = nullptr; const void* scalar_r = nullptr;
  for (int64_t i = 0; i < n_spans; ++i) {
    const ag_span3& sp = spans[i];
    if (sp.n < 0) AG_FAIL(AG_ERR_INVALID, "arith_spans: negative length");
    if (sp.n == 0) continue;
    if (!sp.l || !sp.r || !sp.out) AG_FAIL(AG_ERR_INVALID, "arith_spans: NULL operand");
    if (!la) scalar_l = sp.l;
    if (!ra) scalar_r = sp.r;
    for (int64_t r0 = 0; r0 < sp.n; r0 += chunk) {
      Piece p{(const char*)sp.l + (la ? r0 * w : 0), (const char*)sp.r + (ra ? r0 * w : 0), (char*)sp.out + r0 * w, sp.n - r0 < chunk ? sp.n - r0 : chunk};
      if (!pieces.empty()) {
        Piece& q = pieces.back();
        const bool cont = (!la || q.l + q.n * w == p.l) && (!ra || q.r + q.n * w == p.r) && q.out + q.n * w == p.out;
        if (cont && q.n + p.n <= chunk) { q.n += p.n; continue; }
      }
      pieces.push_back(p);
    }
  }
  if (pieces.empty()) return AG_OK;
  Pipe pipe;
  AG_TRY(pipe.acquire());
  void* d_l[kPipe] = {}; void* d_r[kPipe] = {}; void* d_o[kPipe] = {};
  ag_status rc = AG_OK;
  const size_t stage_bytes = (size_t)(chunk + pad) * w + 64;
  for (int sl = 0; sl < kPipe && rc == AG_OK; ++sl) {
    if (la) rc = dev_alloc_async(&d_l[sl], stage_bytes, pipe.s[sl]);
    if (rc == AG_OK && ra) rc = dev_alloc_async(&d_r[sl], stage_bytes, pipe.s[sl]);
    if (rc == AG_OK) rc = dev_alloc_async(&d_o[sl], stage_bytes, pipe.s[sl]);
  }
  int64_t ci = 0;
  for (size_t first = 0; first < pieces.size() && rc == AG_OK; ++ci) {
    const int sl = (int)(ci % kPipe);
    cudaStream_t st = pipe.s[sl];
    // pieces [first, last) of this stage, each at a 16-byte aligned row offset
    size_t last = first;
    int64_t rows = 0;
    while (last < pieces.size()) {
      const int64_t at = (rows + pad - 1) / pad * pad;
      if (last > first && at + pieces[last].n > chunk) break;
      rows = at + pieces[last].n;
      ++last;
    }
    int64_t at = 0;
    for (size_t k = first; k < last && rc == AG_OK; ++k) {
      at = (at + pad - 1) / pad * pad;
      if (la) rc = h2d((char*)d_l[sl] + at * w, pieces[k].l, (size_t)pieces[k].n * w, st);
      if (rc == AG_OK && ra) rc = h2d((char*)d_r[sl] + at * w, pieces[k].r, (size_t)pieces[k].n * w, st);
      at += pieces[k].n;
    }
    if (rc == AG_OK) rc = arith_binary_dev(type, op, shape, la ? d_l[sl] : scalar_l, ra ? d_r[sl] : scalar_r, d_o[sl], rows, st);
    at = 0;
    for (size_t k = first; k < last && rc == AG_OK; ++k) {
      at = (at + pad - 1) / pad * pad;
      rc = d2h(pieces[k].out, (const char*)d_o[sl] + at * w, (size_t)pieces[k].n * w, st);
      at += pieces[k].n;
    }
    first = last;
  }
  for (int sl = 0; sl < kPipe; ++sl) {
    if (d_l[sl]) cudaFreeAsync(d_l[sl], pipe.s[sl]);
    if (d_r[sl]) cudaFreeAsync(d_r[sl], pipe.s[sl]);
    if (d_o[sl]) cudaFreeAsync(d_o[sl], pipe.s[sl]);
  }
  ag_status rs = pipe.sync_all();
  return rc != AG_OK ? rc : rs;
}

static ag_status host_arith_binary(int type, int8_t op, int shape, const void* l, const void* r, void* out, int64_t n) {
  const int w = type_width(type);
  if (w == 0) AG_FAIL(AG_ERR_TYPE, "arith: unsupported type id %d", type);
  if (n < 0) AG_FAIL(AG_ERR_INVALID, "arith: negative length");
  if (n > 0 && (!l || !r || !out)) AG_FAIL(AG_ERR_INVALID, "arith: NULL operand");
  const void* in[2] = {shape == AG_SHAPE_SA ? nullptr : l, shape == AG_SHAPE_AS ? nullptr : r};
  const int widths[2] = {w, w};
  return pipelined_rows(n, 2, in, widths, out, w, [&](void* const* d_in, void* d_out, int64_t len, cudaStream_t st) {
    return arith_binary_dev(type, op, shape, shape == AG_SHAPE_SA ? l : d_in[0], shape == AG_SHAPE_AS ? r : d_in[1], d_out, len, st);
  });
}

}  // namespace ag

using namespace ag;

extern "C" {

// ---- arithmetic ------------------------------------------------------------------
ag_status ag_arith_binary(int type, int8_t op, const void* l, const void* r, void* out, int64_t n) {
  return host_arith_binary(type, op, AG_SHAPE_AA, l, r, out, n);
}
ag_status ag_arith_arr_scalar(int type, int8_t op, const void* l, const void* r, void* out, int64_t n) {
  return host_arith_binary(type, op, AG_SHAPE_AS, l, r, out, n);
}
ag_status ag_arith_scalar_arr(int type, int8_t op, const void* l, const void* r, void* out, int64_t n) {
  return host_arith_binary(type, op, AG_SHAPE_SA, l, r, out, n);
}
ag_status ag_arith_binary_spans(int type, int8_t op, int shape, const ag_span3* spans, int64_t n_spans) {
  return host_arith_binary_spans(type, op, shape, spans, n_spans);
}
ag_status ag_arith_unary_same(int type, int8_t op, const void* in, void* out, int64_t n) {
  const int w = type_width(type);
  if (w == 0) AG_FAIL(AG_ERR_TYPE, "arith: unsupported type id %d", type);
  if (n < 0) AG_FAIL(AG_ERR_INVALID, "arith: negative length");
  if (n > 0 && (!in || !out)) AG_FAIL(AG_ERR_INVALID, "arith: NULL operand");
  const void* ins[1] = {in};
  const int widths[1] = {w};
  return pipelined_rows(n, 1, ins, widths, out, w, [&](void* const* d_in, void* d_out, int64_t len, cudaStream_t st) {
    return arith_unary_same_dev(type, op, d_in[0], d_out, len, st);
  });
}
ag_status ag_arith_unary_diff(int itype, int otype, int8_t op, const void* in, void* out, int64_t n) {
  const int wi = type_width(itype), wo = type_width(otype);
  if (wi == 0 || wo == 0) AG_FAIL(AG_ERR_TYPE, "arith: unsupported type id");
  if (n < 0) AG_FAIL(AG_ERR_INVALID, "arith: negative length");
  if (n > 0 && (!in || !out)) AG_FAIL(AG_ERR_INVALID, "arith: NULL operand");
  const void* ins[1] = {in};
  const int widths[1] = {wi};
  return pipelined_rows(n, 1, ins, widths, out, wo, [&](void* const* d_in, void* d_out, int64_t len, cudaStream_t st) {
    return arith_unary_diff_dev(itype, otype, op, d_in[0], d_out, len, st);
  });
}

ag_status ag_arith_checked(int type, int8_t op, int shape, const void* l, const uint8_t* lvalid, int64_t loff,
                           const void* r, const uint8_t* rvalid, int64_t roff, void* out, int64_t n, int64_t* first_bad) {
  AG_TRY(ensure_init());
  if (first_bad) *first_bad = AG_NO_ERROR_POS;
  const int w = type_width(type);
  if (w == 0) AG_FAIL(AG_ERR_TYPE, "arith_checked: type id %d is not a numeric type", type);
  if (type_is_float(type) && op != AG_OP_DIV && op != AG_OP_DIV_CHECKED)
    AG_FAIL(AG_ERR_TYPE, "arith_checked: type id %d is not an integer type (floating point types have NotNull kernels for DIV / DIV_CHECKED only)", type);
  if (n < 0) AG_FAIL(AG_ERR_INVALID, "arith_checked: negative length");
  if (n == 0) return AG_OK;
  if ((shape == AG_SHAPE_SA && !l) || (shape == AG_SHAPE_AS && !r)) return AG_OK;  // null scalar
  if (!l || !r || !out) AG_FAIL(AG_ERR_INVALID, "arith_checked: NULL operand");
  CallStream cs;
  AG_TRY(cs.acquire());
  Temps t(cs);
  void *dl = nullptr, *dr = nullptr, *dout = nullptr;
  uint8_t *dlv = nullptr, *drv = nullptr;
  int64_t dloff = 0, droff = 0;
  int64_t* d_bad = nullptr;
  if (shape != AG_SHAPE_SA) { AG_TRY(t.alloc(&dl, (size_t)n * w)); AG_TRY(h2d(dl, l, (size_t)n * w, cs)); AG_TRY(upload_bitmap(t, lvalid, loff, n, &dlv, &dloff)); }
  if (shape != AG_SHAPE_AS) { AG_TRY(t.alloc(&dr, (size_t)n * w)); AG_TRY(h2d(dr, r, (size_t)n * w, cs)); AG_TRY(upload_bitmap(t, rvalid, roff, n, &drv, &droff)); }
  AG_TRY(t.alloc(&dout, (size_t)n * w));
  AG_TRY(t.alloc_t(&d_bad, sizeof(int64_t)));
  AG_TRY(error_word_reset(d_bad, cs));
  AG_TRY(arith_checked_dev(type, op, shape, shape == AG_SHAPE_SA ? l : dl, dlv, dloff, shape == AG_SHAPE_AS ? r : dr, drv, droff, dout, n, d_bad, cs));
  int64_t bad = AG_NO_ERROR_POS;
  AG_TRY(d2h(&bad, d_bad, sizeof(bad), cs));
  AG_TRY(d2h(out, dout, (size_t)n * w, cs));
  AG_TRY(sync(cs));
  if (first_bad) *first_bad = bad;
  if (bad != AG_NO_ERROR_POS) {
    if (op == AG_OP_DIV || op == AG_OP_DIV_CHECKED) AG_FAIL(AG_ERR_INVALID, "divide by zero");  // errDivByZero, base_arithmetic.go:139
    if (op == AG_OP_SHIFT_LEFT_CHECKED || op == AG_OP_SHIFT_RIGHT_CHECKED)
      AG_FAIL(AG_ERR_INVALID, "shift amount must be >= 0 and less than precision of type");     // errShift, scalar_arithmetic.go:294
    AG_FAIL(AG_ERR_INVALID, "overflow");                                                        // errOverflow,  base_arithmetic.go:138
  }
  return AG_OK;
}

ag_status ag_arith_unary_checked(int type, int8_t op, const void* in, void* out, int64_t n, int64_t* first_bad) {
  AG_TRY(ensure_init());
  if (first_bad) *first_bad = AG_NO_ERROR_POS;
  const int w = type_width(type);
  if (w == 0) AG_FAIL(AG_ERR_TYPE, "arith: unsupported type id %d", type);
  if (n < 0) AG_FAIL(AG_ERR_INVALID, "arith: negative length");
  if (n == 0) return AG_OK;
  if (!in || !out) AG_FAIL(AG_ERR_INVALID, "arith: NULL operand");
  CallStream cs; AG_TRY(cs.acquire());
  Temps t(cs);
  void *din, *dout; int64_t* d_bad;
  AG_TRY(t.alloc(&din, (size_t)n * w)); AG_TRY(t.alloc(&dout, (size_t)n * w)); AG_TRY(t.alloc_t(&d_bad, sizeof(int64_t)));
  AG_TRY(h2d(din, in, (size_t)n * w, cs));
  AG_TRY(error_word_reset(d_bad, cs));
  AG_TRY(arith_unary_checked_dev(type, op, din, dout, n, d_bad, cs));
  int64_t bad = AG_NO_ERROR_POS;
  AG_TRY(d2h(&bad, d_bad, sizeof(bad), cs));
  AG_TRY(d2h(out, dout, (size_t)n * w, cs));
  AG_TRY(sync(cs));
  if (first_bad) *first_bad = bad;
  if (bad != AG_NO_ERROR_POS) AG_FAIL(AG_ERR_INVALID, "overflow");
  return AG_OK;
}

// ---- numeric casts -----------------------------------------------------------------
ag_status ag_cast_numeric(int itype, int otype, const void* in, void* out, int64_t n) {
  const int wi = type_width(itype), wo = type_width(otype);
  if (wi == 0 || wo == 0) AG_FAIL(AG_ERR_TYPE, "cast: unsupported type id");
  if (n < 0) AG_FAIL(AG_ERR_INVALID, "cast: negative length");
  if (n > 0 && (!in || !out)) AG_FAIL(AG_ERR_INVALID, "cast: NULL operand");
  const void* ins[1] = {in};
  const int widths[1] = {wi};
  return pipelined_rows(n, 1, ins, widths, out, wo, [&](void* const* d_in, void* d_out, int64_t len, cudaStream_t st) {
    return cast_numeric_dev(itype, otype, d_in[0], nullptr, 0, d_out, len, 1, 1, nullptr, 0, st);
  });
}

ag_status ag_cast_numeric_checked(int itype, int otype, const void* in, const uint8_t* valid, int64_t valid_offset,
                                  void* out, int64_t n, int allow_int_overflow, int allow_float_truncate, int64_t* first_bad) {
  AG_TRY(ensure_init());
  if (first_bad) *first_bad = AG_NO_ERROR_POS;
  const int wi = type_width(itype), wo = type_width(otype);
  if (wi == 0 || wo == 0) AG_FAIL(AG_ERR_TYPE, "cast: unsupported type id");
  if (n < 0 || valid_offset < 0) AG_FAIL(AG_ERR_INVALID, "cast: negative length or offset");
  if (n == 0) return AG_OK;
  if (!in || !out) AG_FAIL(AG_ERR_INVALID, "cast: NULL operand");
  CallStream cs; AG_TRY(cs.acquire());
  Temps t(cs);
  void *din, *dout; int64_t* d_bad; uint8_t* dvalid = nullptr;
  AG_TRY(t.alloc(&din, (size_t)n * wi)); AG_TRY(t.alloc(&dout, (size_t)n * wo)); AG_TRY(t.alloc_t(&d_bad, sizeof(int64_t)));
  AG_TRY(h2d(din, in, (size_t)n * wi, cs));
  const int64_t vbyte0 = valid_offset >> 3;
  if (valid) {
    const size_t vbytes = (size_t)(bytes_for_bits(valid_offset + n) - vbyte0);
    AG_TRY(t.alloc_t(&dvalid, vbytes));
    AG_TRY(h2d(dvalid, valid + vbyte0, vbytes, cs));
  }
  AG_TRY(error_word_reset(d_bad, cs));
  AG_TRY(cast_numeric_dev(itype, otype, din, dvalid, valid_offset & 7, dout, n, allow_int_overflow, allow_float_truncate, d_bad, 0, cs));
  int64_t bad = AG_NO_ERROR_POS;
  AG_TRY(d2h(&bad, d_bad, sizeof(bad), cs));
  AG_TRY(d2h(out, dout, (size_t)n * wo, cs));
  AG_TRY(sync(cs));
  if (first_bad) *first_bad = bad;
  if (bad != AG_NO_ERROR_POS) {
    // numeric_cast.go:614-617 / helpers.go:591-594 wording; the offending element is in the caller's buffer
    if (type_is_float(itype)) {
      const double v = itype == AG_TYPE_FLOAT32 ? (double)((const float*)in)[bad] : ((const double*)in)[bad];
      AG_FAIL(AG_ERR_INVALID, "float value %f was truncated converting to type id %d", v, otype);
    }
    AG_FAIL(AG_ERR_INVALID, "integer value not in range (row %lld)", (long long)bad);
  }
  return AG_OK;
}

// ---- cumulative sum ----------------------------------------------------------------
ag_status ag_cumulative_sum(int type, const void* in, const uint8_t* valid, int64_t valid_offset, int64_t n,
                            const void* start, int skip_nulls, int checked,
                            void* out, uint8_t* out_valid, int64_t* null_count, int64_t* first_bad) {
  AG_TRY(ensure_init());
  if (first_bad) *first_bad = AG_NO_ERROR_POS;
  if (null_count) *null_count = 0;
  const int w = type_width(type);
  if (w == 0) AG_FAIL(AG_ERR_TYPE, "cumulative_sum: input type must be numeric, got type id %d", type);
  if (n < 0 || valid_offset < 0) AG_FAIL(AG_ERR_INVALID, "cumulative_sum: negative length or offset");
  if (n == 0) return AG_OK;
  if (!in || !out) AG_FAIL(AG_ERR_INVALID, "cumulative_sum: NULL operand");
  if (valid && !out_valid) AG_FAIL(AG_ERR_INVALID, "cumulative_sum: an input with a validity bitmap needs an output validity bitmap");
  CallStream cs; AG_TRY(cs.acquire());
  Temps t(cs);
  void *din, *dout; int64_t* d_bad; uint8_t *dvalid = nullptr, *dovalid = nullptr; ag_cumsum_state* dstate;
  AG_TRY(t.alloc(&din, (size_t)n * w)); AG_TRY(t.alloc(&dout, (size_t)n * w)); AG_TRY(t.alloc_t(&d_bad, sizeof(int64_t)));
  AG_TRY(t.alloc_t(&dstate, sizeof(ag_cumsum_state)));
  AG_TRY(h2d(din, in, (size_t)n * w, cs));
  const int64_t vbyte0 = valid_offset >> 3;
  const size_t obytes = (size_t)bytes_for_bits(n);
  if (valid) {
    const size_t vbytes = (size_t)(bytes_for_bits(valid_offset + n) - vbyte0);
    AG_TRY(t.alloc_t(&dvalid, vbytes));
    AG_TRY(h2d(dvalid, valid + vbyte0, vbytes, cs));
  }
  if (out_valid) {
    AG_TRY(t.alloc_t(&dovalid, obytes + 4));
    AG_CUDA_TRY(cudaMemsetAsync(dovalid, 0, obytes + 4, cs));
  }
  AG_TRY(error_word_reset(d_bad, cs));
  AG_TRY(cumulative_sum_state_init(dstate, type, start, cs));
  AG_TRY(cumulative_sum_dev(type, din, dvalid, valid_offset & 7, n, skip_nulls, checked, dout, dovalid, 0, dstate, d_bad, cs));
  int64_t bad = AG_NO_ERROR_POS;
  ag_cumsum_state hs;
  AG_TRY(d2h(&bad, d_bad, sizeof(bad), cs));
  AG_TRY(d2h(&hs, dstate, sizeof(hs), cs));
  AG_TRY(d2h(out, dout, (size_t)n * w, cs));
  if (out_valid) {
    // whole bytes except the last, whose bits past n keep the caller's values
    AG_TRY(sync(cs));
    std::vector<uint8_t> tmp(obytes);
    AG_TRY(d2h(tmp.data(), dovalid, obytes, cs));
    AG_TRY(sync(cs));
    const int tail = (int)(n & 7);
    if (tail) { const uint8_t m = (uint8_t)((1u << tail) - 1u); tmp[obytes - 1] = (uint8_t)((tmp[obytes - 1] & m) | (out_valid[obytes - 1] & ~m)); }
    memcpy(out_valid, tmp.data(), obytes);
  }
  AG_TRY(sync(cs));
  if (first_bad) *first_bad = bad;
  if (null_count) *null_count = hs.null_count;
  if (checked && bad != AG_NO_ERROR_POS) AG_FAIL(AG_ERR_INVALID, "overflow");
  return AG_OK;
}

// ---- comparisons -------------------------------------------------------------------
ag_status ag_compare(int type, int cmp, int shape, const void* l, const void* r, uint8_t* out_bits, int64_t n, int bit_offset) {
  AG_TRY(ensure_init());
  const int w = type_width(type);
  if (w == 0) AG_FAIL(AG_ERR_TYPE, "compare: unsupported type id %d", type);
  if (n < 0) AG_FAIL(AG_ERR_INVALID, "compare: negative length");
  if (n == 0) return AG_OK;
  if (!l || !r || !out_bits) AG_FAIL(AG_ERR_INVALID, "compare: NULL operand");
  const int phase = bit_offset & 7;  // the reference uses offset % 8 relative to `out` (scalar_comparison.cc:72)
  const int64_t out_bytes = (phase + n + 7) >> 3;
  Pipe pipe;
  AG_TRY(pipe.acquire());
  cudaStream_t s0 = pipe.s[0];
  uint8_t* d_bits = nullptr;
  AG_TRY(dev_alloc_async((void**)&d_bits, (size_t)out_bytes + 64, s0));
  ag_status rc = AG_OK;
  // the first and last bytes may hold neighbours' bits that must survive
  rc = h2d(d_bits, out_bits, 1, s0);
  if (rc == AG_OK && out_bytes > 1) rc = h2d(d_bits + out_bytes - 1, out_bits + out_bytes - 1, 1, s0);
  if (rc == AG_OK) rc = sync(s0);
  // chunk boundaries fall on multiples of 1024 output bits, so chunks never share an output word
  int64_t chunk = (kChunkBytes / w) & ~(int64_t)1023;
  const bool la = shape != AG_SHAPE_SA, ra = shape != AG_SHAPE_AS;
  void* d_l[kPipe] = {};
  void* d_r[kPipe] = {};
  for (int sl = 0; sl < kPipe && rc == AG_OK; ++sl) {
    if (la) rc = dev_alloc_async(&d_l[sl], (size_t)chunk * w + 64, pipe.s[sl]);
    if (rc == AG_OK && ra) rc = dev_alloc_async(&d_r[sl], (size_t)chunk * w + 64, pipe.s[sl]);
  }
  int64_t r0 = 0, ci = 0;
  while (r0 < n && rc == AG_OK) {
    int64_t len = (ci == 0) ? (chunk - phase) : chunk;  // (phase + r0) % 1024 == 0 from the second chunk on
    if (len > n - r0) len = n - r0;
    const int sl = (int)(ci % kPipe);
    cudaStream_t st = pipe.s[sl];
    if (la) rc = h2d(d_l[sl], (const char*)l + r0 * w, (size_t)len * w, st);
    if (rc == AG_OK && ra) rc = h2d(d_r[sl], (const char*)r + r0 * w, (size_t)len * w, st);
    const int64_t obit = phase + r0;
    if (rc == AG_OK) rc = compare_dev(type, cmp, shape, la ? d_l[sl] : l, ra ? d_r[sl] : r, d_bits + (obit >> 3), len, (int)(obit & 7), st);
    r0 += len; ++ci;
  }
  for (int sl = 0; sl < kPipe; ++sl) {
    if (d_l[sl]) cudaFreeAsync(d_l[sl], pipe.s[sl]);
    if (d_r[sl]) cudaFreeAsync(d_r[sl], pipe.s[sl]);
  }
  ag_status rs = pipe.sync_all();
  if (rc == AG_OK) rc = rs;
  if (rc == AG_OK) rc = d2h(out_bits, d_bits, (size_t)out_bytes, s0);
  cudaFreeAsync(d_bits, s0);
  rs = sync(s0);
  return rc != AG_OK ? rc : rs;
}

#define AG_CMP_NAMED(NAME, CMP, SHAPE)                                                                        \
  ag_status NAME(int type, const void* l, const void* r, void* out, int64_t n, int offset) {                  \
    return ag_compare(type, CMP, SHAPE, l, r, (uint8_t*)out, n, offset);                                      \
  }
AG_CMP_NAMED(ag_cmp_eq_aa, AG_CMP_EQ, AG_SHAPE_AA) AG_CMP_NAMED(ag_cmp_eq_as, AG_CMP_EQ, AG_SHAPE_AS) AG_CMP_NAMED(ag_cmp_eq_sa, AG_CMP_EQ, AG_SHAPE_SA)
AG_CMP_NAMED(ag_cmp_ne_aa, AG_CMP_NE, AG_SHAPE_AA) AG_CMP_NAMED(ag_cmp_ne_as, AG_CMP_NE, AG_SHAPE_AS) AG_CMP_NAMED(ag_cmp_ne_sa, AG_CMP_NE, AG_SHAPE_SA)
AG_CMP_NAMED(ag_cmp_gt_aa, AG_CMP_GT, AG_SHAPE_AA) AG_CMP_NAMED(ag_cmp_gt_as, AG_CMP_GT, AG_SHAPE_AS) AG_CMP_NAMED(ag_cmp_gt_sa, AG_CMP_GT, AG_SHAPE_SA)
AG_CMP_NAMED(ag_cmp_ge_aa, AG_CMP_GE, AG_SHAPE_AA) AG_CMP_NAMED(ag_cmp_ge_as, AG_CMP_GE, AG_SHAPE_AS) AG_CMP_NAMED(ag_cmp_ge_sa, AG_CMP_GE, AG_SHAPE_SA)
#undef AG_CMP_NAMED

// ---- bitmaps -----------------------------------------------------------------------
// An output bitmap range is staged with its existing first/last bytes so that bits outside
// [off, off+n) survive the round trip; only the bytes of the range are written back.
struct OutBitmap {
  uint8_t* h = nullptr; uint8_t* d = nullptr; int64_t b0 = 0, nbytes = 0, doff = 0;
  ag_status stage(Temps& t, uint8_t* host, int64_t off, int64_t n) {
    h = host; b0 = off >> 3; nbytes = ((off + n + 7) >> 3) - b0; doff = off & 7;
    AG_TRY(t.alloc_t(&d, (size_t)nbytes));
    AG_TRY(h2d(d, h + b0, 1, t.st));
    if (nbytes > 1) AG_TRY(h2d(d + nbytes - 1, h + b0 + nbytes - 1, 1, t.st));
    return AG_OK;
  }
  ag_status fetch(cudaStream_t st) { return d2h(h + b0, d, (size_t)nbytes, st); }
};

ag_status ag_bitmap_op(int bitop, const uint8_t* l, int64_t loff, const uint8_t* r, int64_t roff, uint8_t* out, int64_t ooff, int64_t n) {
  AG_TRY(ensure_init());
  if (n < 0 || loff < 0 || roff < 0 || ooff < 0) AG_FAIL(AG_ERR_INVALID, "bitmap_op: negative length or offset");
  if (n == 0) return AG_OK;
  if (!l || !r || !out) AG_FAIL(AG_ERR_INVALID, "bitmap_op: NULL bitmap");
  CallStream cs; AG_TRY(cs.acquire());
  Temps t(cs);
  uint8_t *dl, *dr; int64_t dlo, dro;
  AG_TRY(upload_bitmap(t, l, loff, n, &dl, &dlo));
  AG_TRY(upload_bitmap(t, r, roff, n, &dr, &dro));
  OutBitmap ob; AG_TRY(ob.stage(t, out, ooff, n));
  AG_TRY(bitmap_op_dev(bitop, dl, dlo, dr, dro, ob.d, ob.doff, n, cs));
  AG_TRY(ob.fetch(cs));
  return sync(cs);
}
static ag_status host_bitmap_copy(const uint8_t* src, int64_t soff, int64_t n, uint8_t* dst, int64_t doff, bool invert) {
  AG_TRY(ensure_init());
  if (n < 0 || soff < 0 || doff < 0) AG_FAIL(AG_ERR_INVALID, "bitmap_copy: negative length or offset");
  if (n == 0) return AG_OK;
  if (!src || !dst) AG_FAIL(AG_ERR_INVALID, "bitmap_copy: NULL bitmap");
  CallStream cs; AG_TRY(cs.acquire());
  Temps t(cs);
  uint8_t* ds; int64_t dso;
  AG_TRY(upload_bitmap(t, src, soff, n, &ds, &dso));
  OutBitmap ob; AG_TRY(ob.stage(t, dst, doff, n));
  AG_TRY(bitmap_copy_dev(ds, dso, n, ob.d, ob.doff, invert, cs));
  AG_TRY(ob.fetch(cs));
  return sync(cs);
}
ag_status ag_bitmap_copy(const uint8_t* src, int64_t soff, int64_t n, uint8_t* dst, int64_t doff) { return host_bitmap_copy(src, soff, n, dst, doff, false); }
ag_status ag_bitmap_invert(const uint8_t* src, int64_t soff, int64_t n, uint8_t* dst, int64_t doff) { return host_bitmap_copy(src, soff, n, dst, doff, true); }
ag_status ag_bitmap_set(uint8_t* bits, int64_t off, int64_t n, int value) {
  AG_TRY(ensure_init());
  if (n < 0 || off < 0) AG_FAIL(AG_ERR_INVALID, "bitmap_set: negative length or offset");
  if (n == 0) return AG_OK;
  if (!bits) AG_FAIL(AG_ERR_INVALID, "bitmap_set: NULL bitmap");
  CallStream cs; AG_TRY(cs.acquire());
  Temps t(cs);
  OutBitmap ob; AG_TRY(ob.stage(t, bits, off, n));
  AG_TRY(bitmap_set_dev(ob.d, ob.doff, n, value, cs));
  AG_TRY(ob.fetch(cs));
  return sync(cs);
}
ag_status ag_bitmap_popcount(const uint8_t* bits, int64_t off, int64_t n, int64_t* count) {
  AG_TRY(ensure_init());
  if (!count) AG_FAIL(AG_ERR_INVALID, "popcount: NULL result");
  *count = 0;
  if (n < 0 || off < 0) AG_FAIL(AG_ERR_INVALID, "popcount: negative length or offset");
  if (n == 0) return AG_OK;
  if (!bits) AG_FAIL(AG_ERR_INVALID, "popcount: NULL bitmap");
  CallStream cs; AG_TRY(cs.acquire());
  Temps t(cs);
  uint8_t* d; int64_t doff; int64_t* d_count;
  AG_TRY(upload_bitmap(t, bits, off, n, &d, &doff));
  AG_TRY(t.alloc_t(&d_count, sizeof(int64_t)));
  AG_TRY(bitmap_popcount_dev(d, doff, n, d_count, cs));
  AG_TRY(d2h(count, d_count, sizeof(int64_t), cs));
  return sync(cs);
}
ag_status ag_kleene(int kop, const uint8_t* lvalid, const uint8_t* ldata, int64_t loff, const uint8_t* rvalid, const uint8_t* rdata, int64_t roff,
                    uint8_t* out_valid, uint8_t* out_data, int64_t ooff, int64_t n) {
  AG_TRY(ensure_init());
  if (n < 0 || loff < 0 || roff < 0 || ooff < 0) AG_FAIL(AG_ERR_INVALID, "kleene: negative length or offset");
  if (n == 0) return AG_OK;
  if (!ldata || !rdata || !out_valid || !out_data) AG_FAIL(AG_ERR_INVALID, "kleene: NULL bitmap");
  CallStream cs; AG_TRY(cs.acquire());
  Temps t(cs);
  uint8_t *dlv, *dld, *drv, *drd; int64_t o1, o2, o3, o4;
  AG_TRY(upload_bitmap(t, lvalid, loff, n, &dlv, &o1));
  AG_TRY(upload_bitmap(t, ldata, loff, n, &dld, &o2));
  AG_TRY(upload_bitmap(t, rvalid, roff, n, &drv, &o3));
  AG_TRY(upload_bitmap(t, rdata, roff, n, &drd, &o4));
  OutBitmap ov, od;
  AG_TRY(ov.stage(t, out_valid, ooff, n));
  AG_TRY(od.stage(t, out_data, ooff, n));
  AG_TRY(kleene_dev(kop, dlv, dld, o2, drv, drd, o4, ov.d, od.d, ov.doff, n, cs));
  AG_TRY(ov.fetch(cs));
  AG_TRY(od.fetch(cs));
  return sync(cs);
}

// ---- filter / take -----------------------------------------------------------------
ag_status ag_filter_output_size(const uint8_t* mask, const uint8_t* mvalid, int64_t moff, int64_t n, int null_selection, int64_t* out_len) {
  AG_TRY(ensure_init());
  if (!out_len) AG_FAIL(AG_ERR_INVALID, "filter_output_size: NULL result");
  *out_len = 0;
  if (n < 0 || moff < 0) AG_FAIL(AG_ERR_INVALID, "filter_output_size: negative length or offset");
  if (n == 0) return AG_OK;
  if (!mask) AG_FAIL(AG_ERR_INVALID, "filter_output_size: NULL mask");
  CallStream cs; AG_TRY(cs.acquire());
  Temps t(cs);
  uint8_t *dm, *dmv; int64_t o1, o2; int64_t* d_len;
  AG_TRY(upload_bitmap(t, mask, moff, n, &dm, &o1));
  AG_TRY(upload_bitmap(t, mvalid, moff, n, &dmv, &o2));
  AG_TRY(t.alloc_t(&d_len, sizeof(int64_t)));
  AG_TRY(filter_output_size_dev(dm, dmv, o1, n, null_selection, d_len, cs));
  AG_TRY(d2h(out_len, d_len, sizeof(int64_t), cs));
  return sync(cs);
}

ag_status ag_filter_primitive(int bit_width, const void* vals, const uint8_t* vvalid, int64_t voff,
                              const uint8_t* mask, const uint8_t* mvalid, int64_t moff, int64_t n, int null_selection,
                              void* out, uint8_t* out_valid, int64_t* out_len, int64_t* out_nulls) {
  AG_TRY(ensure_init());
  if (!out_len) AG_FAIL(AG_ERR_INVALID, "filter: NULL out_len");
  *out_len = 0;
  if (out_nulls) *out_nulls = 0;
  if (n < 0 || moff < 0 || voff < 0) AG_FAIL(AG_ERR_INVALID, "filter: negative length or offset");
  if (bit_width != 1 && bit_width != 8 && bit_width != 16 && bit_width != 32 && bit_width != 64) AG_FAIL(AG_ERR_TYPE, "filter: invalid values bit width %d", bit_width);
  if (n == 0) return AG_OK;
  if (!vals || !mask) AG_FAIL(AG_ERR_INVALID, "filter: NULL values/mask");
  if (bit_width == 1) {  // boolean values: bitmap in, bitmap out
    CallStream cs; AG_TRY(cs.acquire());
    Temps t(cs);
    uint8_t *dm, *dmv, *dvv, *dvd; int64_t om, omv, ovv, ovd; int64_t* d_len;
    AG_TRY(upload_bitmap(t, mask, moff, n, &dm, &om));
    AG_TRY(upload_bitmap(t, mvalid, moff, n, &dmv, &omv));
    AG_TRY(upload_bitmap(t, (const uint8_t*)vals, voff, n, &dvd, &ovd));
    AG_TRY(upload_bitmap(t, vvalid, voff, n, &dvv, &ovv));
    AG_TRY(t.alloc_t(&d_len, 2 * sizeof(int64_t)));
    AG_TRY(filter_output_size_dev(dm, dmv, om, n, null_selection, d_len, cs));
    int64_t len = 0;
    AG_TRY(d2h(&len, d_len, sizeof(int64_t), cs));
    AG_TRY(sync(cs));
    uint8_t *dout, *dov = nullptr;
    AG_TRY(t.alloc_t(&dout, (size_t)((len + 31) / 32) * 4));
    if (out_valid) AG_TRY(t.alloc_t(&dov, (size_t)((len + 31) / 32) * 4));
    // values bitmap and its validity share the row numbering: both copies keep phase voff & 7
    AG_TRY(filter_primitive_dev(1, dvd, dvv, ovd, dm, dmv, om, n, null_selection, dout, dov, len, d_len + 1, cs));
    AG_TRY(d2h(out, dout, (size_t)((len + 7) / 8), cs));
    if (out_valid) AG_TRY(d2h(out_valid, dov, (size_t)((len + 7) / 8), cs));
    int64_t valid = 0;
    if (out_valid && out_nulls) {
      AG_TRY(bitmap_popcount_dev(dov, 0, len, d_len, cs));
      AG_TRY(d2h(&valid, d_len, sizeof(int64_t), cs));
    }
    AG_TRY(sync(cs));
    *out_len = len;
    if (out_valid && out_nulls) *out_nulls = len - valid;
    return AG_OK;
  }
  const int w = bit_width / 8;
  CallStream cs; AG_TRY(cs.acquire());
  Temps t(cs);
  uint8_t *dm, *dmv, *dvv; int64_t om, omv, ovv; int64_t* d_len;
  AG_TRY(upload_bitmap(t, mask, moff, n, &dm, &om));
  AG_TRY(upload_bitmap(t, mvalid, moff, n, &dmv, &omv));
  AG_TRY(t.alloc_t(&d_len, 2 * sizeof(int64_t)));
  // pass 1 over the mask (getFilterOutputSize) while the values are still in flight
  AG_TRY(filter_output_size_dev(dm, dmv, om, n, null_selection, d_len, cs));
  int64_t len = 0;
  AG_TRY(d2h(&len, d_len, sizeof(int64_t), cs));
  void* dv; AG_TRY(t.alloc(&dv, (size_t)n * w));
  AG_TRY(h2d(dv, (const char*)vals + voff * w, (size_t)n * w, cs));
  AG_TRY(upload_bitmap(t, vvalid, voff, n, &dvv, &ovv));
  AG_TRY(sync(cs));
  void* dout; AG_TRY(t.alloc(&dout, (size_t)len * w));
  uint8_t* dov = nullptr;
  if (out_valid) AG_TRY(t.alloc_t(&dov, (size_t)((len + 31) / 32) * 4));
  // the device copy of the values starts at the slice: element offset 0, validity phase ovv
  // (the kernel indexes values and their validity with the same row number, so shift the
  // validity pointer/offset instead of the values)
  AG_TRY(filter_primitive_dev(bit_width, (const char*)dv - ovv * w, dvv, ovv, dm, dmv, om, n, null_selection, dout, dov, len, d_len + 1, cs));
  AG_TRY(d2h(out, dout, (size_t)len * w, cs));
  if (out_valid) AG_TRY(d2h(out_valid, dov, (size_t)((len + 7) / 8), cs));
  int64_t nulls = 0;
  if (out_valid && out_nulls) {
    AG_TRY(bitmap_popcount_dev(dov, 0, len, d_len, cs));
    AG_TRY(d2h(&nulls, d_len, sizeof(int64_t), cs));
  }
  AG_TRY(sync(cs));
  *out_len = len;
  if (out_valid && out_nulls) *out_nulls = len - nulls;
  return AG_OK;
}

ag_status ag_take_indices(int index_width, const uint8_t* mask, const uint8_t* mvalid, int64_t moff, int64_t n,
                          int null_selection, void* out_idx, uint8_t* out_valid, int64_t* out_len) {
  AG_TRY(ensure_init());
  if (!out_len) AG_FAIL(AG_ERR_INVALID, "take_indices: NULL out_len");
  *out_len = 0;
  if (n < 0 || moff < 0) AG_FAIL(AG_ERR_INVALID, "take_indices: negative length or offset");
  if (index_width != 16 && index_width != 32) AG_FAIL(AG_ERR_TYPE, "take_indices: index width must be 16 or 32");
  if (n == 0) return AG_OK;
  if (!mask) AG_FAIL(AG_ERR_INVALID, "take_indices: NULL mask");
  const int w = index_width / 8;
  CallStream cs; AG_TRY(cs.acquire());
  Temps t(cs);
  uint8_t *dm, *dmv; int64_t om, omv; int64_t* d_len;
  AG_TRY(upload_bitmap(t, mask, moff, n, &dm, &om));
  AG_TRY(upload_bitmap(t, mvalid, moff, n, &dmv, &omv));
  AG_TRY(t.alloc_t(&d_len, 2 * sizeof(int64_t)));
  AG_TRY(filter_output_size_dev(dm, dmv, om, n, null_selection, d_len, cs));
  int64_t len = 0;
  AG_TRY(d2h(&len, d_len, sizeof(int64_t), cs));
  AG_TRY(sync(cs));
  void* dout; AG_TRY(t.alloc(&dout, (size_t)len * w));
  uint8_t* dov = nullptr;
  if (out_valid) AG_TRY(t.alloc_t(&dov, (size_t)((len + 31) / 32) * 4));
  AG_TRY(take_indices_dev(index_width, dm, dmv, om, n, null_selection, dout, dov, len, d_len + 1, cs));
  AG_TRY(d2h(out_idx, dout, (size_t)len * w, cs));
  if (out_valid) AG_TRY(d2h(out_valid, dov, (size_t)((len + 7) / 8), cs));
  AG_TRY(sync(cs));
  *out_len = len;
  return AG_OK;
}

ag_status ag_take_primitive(int bit_width, const void* vals, const uint8_t* vvalid, int64_t voff, int64_t vlen,
                            int idx_width, int idx_signed, const void* idx, const uint8_t* ivalid, int64_t ioff,
                            int64_t n, int bounds_check, void* out, uint8_t* out_valid,
                            int64_t* out_nulls, int64_t* bad_pos, int64_t* bad_index) {
  AG_TRY(ensure_init());
  if (bad_pos) *bad_pos = AG_NO_ERROR_POS;
  if (out_nulls) *out_nulls = 0;
  if (n < 0 || voff < 0 || ioff < 0 || vlen < 0) AG_FAIL(AG_ERR_INVALID, "take: negative length or offset");
  if (bit_width != 1 && bit_width != 8 && bit_width != 16 && bit_width != 32 && bit_width != 64) AG_FAIL(AG_ERR_INVALID, "take: invalid values byte width for take");
  if (idx_width != 8 && idx_width != 16 && idx_width != 32 && idx_width != 64) AG_FAIL(AG_ERR_INDEX, "take: invalid indices byte width");
  if (n == 0) return AG_OK;
  if (!idx || !out) AG_FAIL(AG_ERR_INVALID, "take: NULL indices/output");
  const bool is_bool = bit_width == 1;
  const int w = is_bool ? 0 : bit_width / 8, iw = idx_width / 8;
  CallStream cs; AG_TRY(cs.acquire());
  Temps t(cs);
  void *dv, *di, *dout; uint8_t *dvv, *div; int64_t ovv, oiv; int64_t* d_word;
  if (is_bool) {
    uint8_t* dvb; int64_t ovb;
    AG_TRY(upload_bitmap(t, (const uint8_t*)vals, voff, vlen, &dvb, &ovb));
    dv = dvb;
  } else {
    AG_TRY(t.alloc(&dv, (size_t)vlen * w));
    AG_TRY(h2d(dv, (const char*)vals + voff * w, (size_t)vlen * w, cs));
  }
  AG_TRY(upload_bitmap(t, vvalid, voff, vlen, &dvv, &ovv));
  if (is_bool && !vvalid) ovv = voff & 7;
  AG_TRY(t.alloc(&di, (size_t)n * iw));
  AG_TRY(h2d(di, idx, (size_t)n * iw, cs));
  AG_TRY(upload_bitmap(t, ivalid, ioff, n, &div, &oiv));
  AG_TRY(t.alloc(&dout, is_bool ? (size_t)((n + 31) / 32) * 4 : (size_t)n * w));
  uint8_t* dov = nullptr;
  if (out_valid) AG_TRY(t.alloc_t(&dov, (size_t)((n + 31) / 32) * 4));
  AG_TRY(t.alloc_t(&d_word, 2 * sizeof(int64_t)));
  AG_TRY(error_word_reset(d_word, cs));
  // the device copies start at the slice: element offset becomes the bitmap phase (voff & 7)
  AG_TRY(take_primitive_dev(bit_width, is_bool ? dv : (void*)((const char*)dv - ovv * w), dvv, ovv, vlen, idx_width, idx_signed, di, div, oiv, n,
                            bounds_check, dout, dov, d_word, cs));
  int64_t bad = AG_NO_ERROR_POS;
  AG_TRY(d2h(&bad, d_word, sizeof(int64_t), cs));
  AG_TRY(sync(cs));
  if (bad != AG_NO_ERROR_POS) {
    if (bad_pos) *bad_pos = bad;
    int64_t v = 0;
    switch (idx_width) {
      case 8: v = idx_signed ? (int64_t)((const int8_t*)idx)[bad] : (int64_t)((const uint8_t*)idx)[bad]; break;
      case 16: v = idx_signed ? (int64_t)((const int16_t*)idx)[bad] : (int64_t)((const uint16_t*)idx)[bad]; break;
      case 32: v = idx_signed ? (int64_t)((const int32_t*)idx)[bad] : (int64_t)((const uint32_t*)idx)[bad]; break;
      default: v = ((const int64_t*)idx)[bad]; break;
    }
    if (bad_index) *bad_index = v;
    if (idx_width == 64 && !idx_signed) AG_FAIL(AG_ERR_INDEX, "%llu out of bounds", (unsigned long long)v);
    AG_FAIL(AG_ERR_INDEX, "%lld out of bounds", (long long)v);  // helpers.go:951
  }
  AG_TRY(d2h(out, dout, is_bool ? (size_t)((n + 7) / 8) : (size_t)n * w, cs));
  if (out_valid) {
    AG_TRY(d2h(out_valid, dov, (size_t)((n + 7) / 8), cs));
    if (out_nulls) {
      AG_TRY(bitmap_popcount_dev(dov, 0, n, d_word + 1, cs));
      int64_t valid = 0;
      AG_TRY(d2h(&valid, d_word + 1, sizeof(int64_t), cs));
      AG_TRY(sync(cs));
      *out_nulls = n - valid;
      return AG_OK;
    }
  }
  return sync(cs);
}

ag_status ag_sort_indices(int type, const void* vals, const uint8_t* valid, int64_t offset, int64_t n, int order,
                          int null_placement, uint64_t* out, int64_t* null_count, int64_t* nan_count) {
  AG_TRY(ensure_init());
  if (null_count) *null_count = 0;
  if (nan_count) *nan_count = 0;
  const int w = type_width(type);
  if (w == 0) AG_FAIL(AG_ERR_NOT_IMPLEMENTED, "sort_indices: unsupported type id %d (fixed-width numeric columns only)", type);
  if (n < 0 || offset < 0) AG_FAIL(AG_ERR_INVALID, "sort_indices: negative length or offset");
  if (n == 0) return AG_OK;
  if (!vals || !out) AG_FAIL(AG_ERR_INVALID, "sort_indices: NULL values/output");
  CallStream cs; AG_TRY(cs.acquire());
  Temps t(cs);
  void* dv; uint8_t* dvalid; int64_t ov; uint64_t* dout;
  AG_TRY(t.alloc(&dv, (size_t)n * w));
  AG_TRY(h2d(dv, (const char*)vals + offset * w, (size_t)n * w, cs));
  AG_TRY(upload_bitmap(t, valid, offset, n, &dvalid, &ov));
  AG_TRY(t.alloc_t(&dout, (size_t)n * 8));
  // the device copy starts at the slice: the element offset becomes the bitmap phase (offset & 7)
  AG_TRY(sort_indices_dev(type, (const char*)dv - ov * w, dvalid, ov, n, order, null_placement, dout, null_count, nan_count, cs));
  AG_TRY(d2h(out, dout, (size_t)n * 8, cs));
  return sync(cs);
}

ag_status ag_is_in(int bit_width, const void* vals, const uint8_t* valid, int64_t offset, int64_t n, const void* set_vals,
                   const uint8_t* set_valid, int64_t set_offset, int64_t set_n, int null_behavior, uint8_t* out_data, uint8_t* out_valid,
                   int64_t* out_nulls) {
  AG_TRY(ensure_init());
  if (out_nulls) *out_nulls = 0;
  if (bit_width != 8 && bit_width != 16 && bit_width != 32 && bit_width != 64) AG_FAIL(AG_ERR_NOT_IMPLEMENTED, "is_in: fixed-width values of 1/2/4/8 bytes only");
  if (n < 0 || set_n < 0 || offset < 0 || set_offset < 0) AG_FAIL(AG_ERR_INVALID, "is_in: negative length or offset");
  if (n == 0) return AG_OK;
  if (!vals || !out_data || (set_n > 0 && !set_vals)) AG_FAIL(AG_ERR_INVALID, "is_in: NULL values / value set / output");
  const int w = bit_width / 8;
  CallStream cs; AG_TRY(cs.acquire());
  Temps t(cs);
  void *dv, *ds = nullptr; uint8_t *dvv, *dsv = nullptr, *dod, *dov; int64_t ov, os = 0; int64_t* d_nulls;
  AG_TRY(t.alloc(&dv, (size_t)n * w));
  AG_TRY(h2d(dv, (const char*)vals + offset * w, (size_t)n * w, cs));
  AG_TRY(upload_bitmap(t, valid, offset, n, &dvv, &ov));
  if (set_n > 0) {
    AG_TRY(t.alloc(&ds, (size_t)set_n * w));
    AG_TRY(h2d(ds, (const char*)set_vals + set_offset * w, (size_t)set_n * w, cs));
    AG_TRY(upload_bitmap(t, set_valid, set_offset, set_n, &dsv, &os));
  }
  const size_t bm = (size_t)((n + 31) / 32) * 4;
  AG_TRY(t.alloc_t(&dod, bm));
  AG_TRY(t.alloc_t(&dov, bm));
  AG_TRY(t.alloc_t(&d_nulls, 8));
  AG_TRY(is_in_dev(bit_width, (const char*)dv - ov * w, dvv, ov, n, ds ? (const char*)ds - os * w : nullptr, dsv, os, set_n, null_behavior, dod,
                   out_valid ? dov : nullptr, d_nulls, cs));
  AG_TRY(d2h(out_data, dod, (size_t)((n + 7) / 8), cs));
  if (out_valid) AG_TRY(d2h(out_valid, dov, (size_t)((n + 7) / 8), cs));
  int64_t nulls = 0;
  AG_TRY(d2h(&nulls, d_nulls, 8, cs));
  AG_TRY(sync(cs));
  if (out_nulls) *out_nulls = nulls;
  return AG_OK;
}

ag_status ag_unique(int bit_width, const void* vals, const uint8_t* valid, int64_t offset, int64_t n, void* out, uint8_t* out_valid,
                    int64_t* out_len, int64_t* out_nulls) {
  AG_TRY(ensure_init());
  if (!out_len) AG_FAIL(AG_ERR_INVALID, "unique: NULL out_len");
  *out_len = 0;
  if (out_nulls) *out_nulls = 0;
  if (bit_width != 8 && bit_width != 16 && bit_width != 32 && bit_width != 64) AG_FAIL(AG_ERR_NOT_IMPLEMENTED, "unique: fixed-width values of 1/2/4/8 bytes only");
  if (n < 0 || offset < 0) AG_FAIL(AG_ERR_INVALID, "unique: negative length or offset");
  if (n == 0) return AG_OK;
  if (!vals || !out) AG_FAIL(AG_ERR_INVALID, "unique: NULL values/output");
  if (valid && !out_valid) AG_FAIL(AG_ERR_INVALID, "unique: an input with a validity bitmap needs an output validity bitmap");
  const int w = bit_width / 8;
  CallStream cs; AG_TRY(cs.acquire());
  Temps t(cs);
  void *dv, *dout; uint8_t *dvv, *dov = nullptr; int64_t ov; int64_t* d_len;
  AG_TRY(t.alloc(&dv, (size_t)n * w));
  AG_TRY(h2d(dv, (const char*)vals + offset * w, (size_t)n * w, cs));
  AG_TRY(upload_bitmap(t, valid, offset, n, &dvv, &ov));
  AG_TRY(t.alloc(&dout, (size_t)n * w));
  if (valid) AG_TRY(t.alloc_t(&dov, (size_t)((n + 31) / 32) * 4));
  AG_TRY(t.alloc_t(&d_len, 16));
  AG_TRY(unique_dev(bit_width, (const char*)dv - ov * w, dvv, ov, n, dout, dov, n, d_len, cs));
  int64_t len = 0;
  AG_TRY(d2h(&len, d_len, 8, cs));
  AG_TRY(sync(cs));
  AG_TRY(d2h(out, dout, (size_t)len * w, cs));
  if (dov && out_valid) {
    AG_TRY(d2h(out_valid, dov, (size_t)((len + 7) / 8), cs));
    if (out_nulls) {
      AG_TRY(bitmap_popcount_dev(dov, 0, len, d_len + 1, cs));
      int64_t v = 0;
      AG_TRY(d2h(&v, d_len + 1, 8, cs));
      AG_TRY(sync(cs));
      *out_nulls = len - v;
    }
  }
  AG_TRY(sync(cs));
  *out_len = len;
  return AG_OK;
}

ag_status ag_dictionary_encode(int bit_width, const void* vals, const uint8_t* valid, int64_t offset, int64_t n, int null_encoding, int32_t* indices,
                               uint8_t* indices_valid, void* dict, uint8_t* dict_valid, int64_t* dict_len, int64_t* index_nulls) {
  AG_TRY(ensure_init());
  if (!dict_len) AG_FAIL(AG_ERR_INVALID, "dictionary_encode: NULL dict_len");
  *dict_len = 0;
  if (index_nulls) *index_nulls = 0;
  if (bit_width != 8 && bit_width != 16 && bit_width != 32 && bit_width != 64) AG_FAIL(AG_ERR_NOT_IMPLEMENTED, "dictionary_encode: fixed-width values of 1/2/4/8 bytes only");
  if (n < 0 || offset < 0) AG_FAIL(AG_ERR_INVALID, "dictionary_encode: negative length or offset");
  if (null_encoding != AG_NULL_ENCODING_MASK && null_encoding != AG_NULL_ENCODING_ENCODE)
    AG_FAIL(AG_ERR_INVALID, "dictionary_encode: invalid null encoding behavior %d", null_encoding);
  if (n == 0) return AG_OK;
  if (!vals || !indices || !dict) AG_FAIL(AG_ERR_INVALID, "dictionary_encode: NULL values / indices / dictionary");
  if (valid && null_encoding == AG_NULL_ENCODING_MASK && !indices_valid)
    AG_FAIL(AG_ERR_INVALID, "dictionary_encode: an input with a validity bitmap needs an indices validity bitmap in mask mode");
  if (valid && null_encoding == AG_NULL_ENCODING_ENCODE && !dict_valid)
    AG_FAIL(AG_ERR_INVALID, "dictionary_encode: an input with a validity bitmap needs a dictionary validity bitmap in encode mode");
  const int w = bit_width / 8;
  CallStream cs; AG_TRY(cs.acquire());
  Temps t(cs);
  void *dv, *ddict; uint8_t *dvv, *div = nullptr, *ddv = nullptr; int64_t ov; int32_t* didx; int64_t* d_counts;
  AG_TRY(t.alloc(&dv, (size_t)n * w));
  AG_TRY(h2d(dv, (const char*)vals + offset * w, (size_t)n * w, cs));
  AG_TRY(upload_bitmap(t, valid, offset, n, &dvv, &ov));
  AG_TRY(t.alloc_t(&didx, (size_t)n * 4));
  AG_TRY(t.alloc(&ddict, (size_t)n * w));
  const size_t bm = (size_t)((n + 31) / 32) * 4;
  if (indices_valid) AG_TRY(t.alloc_t(&div, bm));
  if (dict_valid) AG_TRY(t.alloc_t(&ddv, bm));
  AG_TRY(t.alloc_t(&d_counts, 16));
  AG_TRY(dictionary_encode_dev(bit_width, (const char*)dv - ov * w, dvv, ov, n, null_encoding, didx, div, ddict, ddv, n, d_counts, cs));
  int64_t counts[2] = {0, 0};
  AG_TRY(d2h(counts, d_counts, 16, cs));
  AG_TRY(sync(cs));
  AG_TRY(d2h(indices, didx, (size_t)n * 4, cs));
  if (div) AG_TRY(d2h(indices_valid, div, (size_t)((n + 7) / 8), cs));
  AG_TRY(d2h(dict, ddict, (size_t)counts[0] * w, cs));
  if (ddv) AG_TRY(d2h(dict_valid, ddv, (size_t)((counts[0] + 7) / 8), cs));
  AG_TRY(sync(cs));
  *dict_len = counts[0];
  if (index_nulls) *index_nulls = counts[1];
  return AG_OK;
}

}  // extern "C"
