// Score file text in HBM: the rows of the score file and of the .U.log / .Q.log files, formatted
// from the scoring results by the device (score(..., write="device")); see sai_format_input in
// include/sai_b200.h for the row layout.
//
// Each text is a length pass, an exclusive scan of the lengths and a write pass, so that its size is
// known exactly before it is written.  Score rows take one thread each (a row has a bounded number of
// fields).  A log row lists a window's candidates, thousands in a dense window: the digit lengths of
// every candidate are computed and scanned first, so a row's length is two reads of that scan and
// every candidate's place in the row is known on its own; a warp writes a row, its lanes the
// candidates.
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"
#include "format_double.cuh"
#include "format_kernels.cuh"
#include "scratch.cuh"

namespace sai {
namespace {

using fmt::format_double;
using fmt::format_int64;

size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

struct FmtArgs {
  int64_t n_blocks, n_rows;
  const int64_t* block_rows;
  const int64_t* block_str;
  const char* strings;
  const int64_t *start, *end;
  const int32_t* nsnps;
  const int64_t *u, *u_start;
  const double* q;
  const int64_t* q_start;
  const int32_t* q_cnt;
  const int32_t *u_cand, *q_cand;
  const int64_t *u_pref, *q_pref;  // exclusive scans of the candidates' digit lengths, [n + 1]
  const int32_t* field;
  const double* vals;
  int32_t n_fields, n_vals;
};

// ---- candidates: digit lengths --------------------------------------------------------------------
__global__ void k_cand_digits(const int32_t* __restrict__ cand, int64_t n, int64_t* len) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    len[i] = fmt::int64_length(cand[i]);
}

// ---- rows -----------------------------------------------------------------------------------------
__device__ inline int64_t block_of(const FmtArgs& a, int64_t r) {
  int64_t lo = 0, hi = a.n_blocks - 1;  // the last block whose first row is <= r
  while (lo < hi) {
    const int64_t mid = (lo + hi + 1) >> 1;
    if (a.block_rows[mid] <= r) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// Appends to out (or only counts, out == nullptr).
struct Text {
  char* out;
  int64_t n = 0;
  __device__ void put(const char* s, int64_t len) {
    if (out)
      for (int64_t i = 0; i < len; ++i) out[n + i] = s[i];
    n += len;
  }
  __device__ void ch(char c) {
    if (out) out[n] = c;
    ++n;
  }
  __device__ void int64(int64_t v) {
    char buf[24];
    put(buf, format_int64(v, buf));
  }
  __device__ void real(double v) {
    char buf[fmt::kMaxDoubleChars];
    put(buf, format_double(v, buf));
  }
};

__device__ int64_t score_row(const FmtArgs& a, int64_t r, char* out) {
  const int64_t b = block_of(a, r);
  const int64_t* bs = a.block_str + 4 * b;
  Text t{out};
  t.put(a.strings + bs[0], bs[1]);
  t.ch('\t');
  t.int64(a.start[r]);
  t.ch('\t');
  t.int64(a.end[r]);
  t.ch('\t');
  t.put(a.strings + bs[2], bs[3]);
  t.ch('\t');
  const int32_t nsnps = a.nsnps[r];
  t.int64(nsnps);
  t.ch('\t');
  for (int f = 0; f < a.n_fields; ++f) {
    if (f) t.ch('\t');
    const int32_t k = a.field[f];
    if (nsnps == 0) t.put("nan", 3);
    else if (k == SAI_FMT_U) t.int64(a.u[r]);
    else if (k == SAI_FMT_Q) t.real(a.q[r]);
    else t.real(a.vals[r * a.n_vals + k]);
  }
  t.ch('\n');
  return t.n;
}

__global__ void k_row_len(FmtArgs a, int64_t* len) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < a.n_rows; r += (int64_t)gridDim.x * blockDim.x)
    len[r] = score_row(a, r, nullptr);
}

__global__ void k_row_write(FmtArgs a, const int64_t* __restrict__ off, char* text) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < a.n_rows; r += (int64_t)gridDim.x * blockDim.x)
    score_row(a, r, text + off[r]);
}

// ---- log rows -------------------------------------------------------------------------------------
// the window's candidates: *first, and how many (0 prints "NA")
template <bool kU>
__device__ inline int64_t log_cands(const FmtArgs& a, int64_t r, int64_t* first) {
  if (a.nsnps[r] == 0) return 0;
  if constexpr (kU) {
    *first = a.u_start[r];
    return a.u[r];
  } else {
    if (isnan(a.q[r])) return 0;
    *first = a.q_start[r];
    return a.q_cnt[r];
  }
}

// "chrom\tstart\tend\t"
__device__ inline int64_t log_head(const FmtArgs& a, int64_t r, const int64_t* bs, char* out) {
  Text t{out};
  t.put(a.strings + bs[0], bs[1]);
  t.ch('\t');
  t.int64(a.start[r]);
  t.ch('\t');
  t.int64(a.end[r]);
  t.ch('\t');
  return t.n;
}

template <bool kU>
__global__ void k_log_len(FmtArgs a, int64_t* len) {
  const int64_t* pref = kU ? a.u_pref : a.q_pref;
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < a.n_rows; r += (int64_t)gridDim.x * blockDim.x) {
    const int64_t* bs = a.block_str + 4 * block_of(a, r);
    int64_t s0 = 0;
    const int64_t cnt = log_cands<kU>(a, r, &s0);
    // every candidate is "chrom:pos" and a ',' or the final '\n'
    len[r] = log_head(a, r, bs, nullptr) + (cnt ? cnt * (bs[1] + 2) + pref[s0 + cnt] - pref[s0] : 3);
  }
}

// one warp per row: lane 0 the head, the lanes the candidates
template <bool kU>
__global__ void __launch_bounds__(256) k_log_write(FmtArgs a, const int64_t* __restrict__ off, char* text) {
  const int32_t* cand = kU ? a.u_cand : a.q_cand;
  const int64_t* pref = kU ? a.u_pref : a.q_pref;
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < a.n_rows; r += warps) {
    const int64_t* bs = a.block_str + 4 * block_of(a, r);
    char* out = text + off[r];
    int64_t s0 = 0;
    const int64_t cnt = log_cands<kU>(a, r, &s0);
    const int64_t head = log_head(a, r, bs, lane == 0 ? out : nullptr);
    if (cnt == 0) {
      if (lane == 0) {
        out[head] = 'N';
        out[head + 1] = 'A';
        out[head + 2] = '\n';
      }
      continue;
    }
    const char* chrom = a.strings + bs[0];
    const int64_t clen = bs[1];
    for (int64_t k = s0 + lane; k < s0 + cnt; k += 32) {
      Text t{out + head + (k - s0) * (clen + 2) + (pref[k] - pref[s0])};
      t.put(chrom, clen);
      t.ch(':');
      t.int64(cand[k]);
      t.ch(k + 1 < s0 + cnt ? ',' : '\n');
    }
  }
}

__global__ void k_format_doubles(const double* __restrict__ x, int64_t n, char* out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    char buf[fmt::kMaxDoubleChars] = {};
    format_double(x[i], buf);
    memcpy(out + 32 * i, buf, 32);
  }
}

// every pointer and range the kernels will read
int check_input(const sai_format_input* in, bool* has_u, bool* has_q) {
  SAI_REQUIRE(in, "sai_engine_format_scores: NULL input");
  const int64_t nb = in->n_blocks, n = in->n_rows;
  SAI_REQUIRE(nb >= 0 && n >= 0 && in->n_fields >= 0 && in->n_vals >= 0 && in->strings_len >= 0 &&
                  in->n_u_cand >= 0 && in->n_q_cand >= 0,
              "sai_engine_format_scores: negative size");
  SAI_REQUIRE(n == 0 || nb > 0, "sai_engine_format_scores: %lld rows in no block", (long long)n);
  if (nb > 0) {
    SAI_REQUIRE(in->block_rows && in->block_str && (in->strings || in->strings_len == 0), "sai_engine_format_scores: NULL blocks");
    SAI_REQUIRE(in->block_rows[0] == 0 && in->block_rows[nb] == n, "sai_engine_format_scores: blocks do not cover the rows");
    for (int64_t b = 0; b < nb; ++b) {
      SAI_REQUIRE(in->block_rows[b] <= in->block_rows[b + 1], "sai_engine_format_scores: block %lld ends before it starts",
                  (long long)b);
      const int64_t* s = in->block_str + 4 * b;
      SAI_REQUIRE(s[0] >= 0 && s[1] >= 0 && s[0] + s[1] <= in->strings_len && s[2] >= 0 && s[3] >= 0 &&
                      s[2] + s[3] <= in->strings_len,
                  "sai_engine_format_scores: block %lld's strings are outside `strings`", (long long)b);
    }
  }
  SAI_REQUIRE(in->n_fields == 0 || in->field, "sai_engine_format_scores: NULL fields");
  *has_u = *has_q = false;
  for (int f = 0; f < in->n_fields; ++f) {
    const int32_t k = in->field[f];
    SAI_REQUIRE(k == SAI_FMT_U || k == SAI_FMT_Q || (k >= 0 && k < in->n_vals),
                "sai_engine_format_scores: field %d is %d (U, Q or a column 0..%d)", f, k, in->n_vals - 1);
    *has_u |= k == SAI_FMT_U;
    *has_q |= k == SAI_FMT_Q;
  }
  if (n == 0) return SAI_OK;
  SAI_REQUIRE(in->start && in->end && in->nsnps, "sai_engine_format_scores: NULL window columns");
  SAI_REQUIRE(in->n_vals == 0 || in->vals, "sai_engine_format_scores: NULL values");
  if (*has_u) {
    SAI_REQUIRE(in->u && in->u_start && (in->u_cand || in->n_u_cand == 0), "sai_engine_format_scores: NULL U columns");
    for (int64_t r = 0; r < n; ++r)
      SAI_REQUIRE(in->nsnps[r] == 0 || (in->u[r] >= 0 && in->u_start[r] >= 0 && in->u_start[r] + in->u[r] <= in->n_u_cand),
                  "sai_engine_format_scores: row %lld's U candidates are outside u_cand", (long long)r);
  }
  if (*has_q) {
    SAI_REQUIRE(in->q && in->q_start && in->q_cnt && (in->q_cand || in->n_q_cand == 0),
                "sai_engine_format_scores: NULL Q columns");
    for (int64_t r = 0; r < n; ++r)
      SAI_REQUIRE(in->nsnps[r] == 0 || in->q[r] != in->q[r] ||
                      (in->q_cnt[r] >= 0 && in->q_start[r] >= 0 && in->q_start[r] + in->q_cnt[r] <= in->n_q_cand),
                  "sai_engine_format_scores: row %lld's Q candidates are outside q_cand", (long long)r);
  }
  return SAI_OK;
}

}  // namespace

// ---- shared with table_kernels.cu: the int64 length scan and grow-only buffers ---------------------
__global__ void __launch_bounds__(1024) k_len_count(const int64_t* __restrict__ v, int64_t n, int64_t* chunk_sum) {
  for (int64_t c = blockIdx.x; c * 1024 < n; c += gridDim.x) {
    const int64_t i = c * 1024 + threadIdx.x;
    int64_t total;
    block_excl_scan64(i < n ? v[i] : 0, &total);
    if (threadIdx.x == 0) chunk_sum[c] = total;
  }
}

__global__ void __launch_bounds__(1024) k_len_scan(int64_t* chunk, int64_t n_chunks, int64_t* total) {
  int64_t carry = 0;
  for (int64_t base = 0; base < n_chunks; base += blockDim.x) {
    const int64_t i = base + threadIdx.x;
    const int64_t v = i < n_chunks ? chunk[i] : 0;
    int64_t sum;
    const int64_t ex = block_excl_scan64(v, &sum);
    if (i < n_chunks) chunk[i] = carry + ex;
    carry += sum;
  }
  if (threadIdx.x == 0) *total = carry;
}

__global__ void __launch_bounds__(1024) k_len_excl(int64_t* v, int64_t n, const int64_t* __restrict__ chunk_off) {
  for (int64_t c = blockIdx.x; c * 1024 < n; c += gridDim.x) {
    const int64_t i = c * 1024 + threadIdx.x;
    int64_t total;
    const int64_t ex = chunk_off[c] + block_excl_scan64(i < n ? v[i] : 0, &total);
    if (i < n) v[i] = ex;
  }
}

int grid_for(int64_t items, int per_block) {
  const int64_t b = (items + per_block - 1) / per_block;
  return (int)(b < 1 ? 1 : b > 8LL * sm_count() ? 8LL * sm_count() : b);
}

// v[0 .. n) -> exclusive offsets, v[n] = total; chunk: (n + 1023) / 1024 int64 of scratch
void scan_lengths(int64_t* v, int64_t n, int64_t* chunk, cudaStream_t st) {
  const int64_t n_chunks = (n + 1023) / 1024;
  const int grid = grid_for(n, 1024);
  if (n > 0) k_len_count<<<grid, 1024, 0, st>>>(v, n, chunk);
  k_len_scan<<<1, 1024, 0, st>>>(chunk, n_chunks, v + n);
  if (n > 0) k_len_excl<<<grid, 1024, 0, st>>>(v, n, chunk);
}

int grow_dev(void** p, size_t* cap, size_t bytes) {
  if (bytes <= *cap) return SAI_OK;
  if (*p) SAI_CUDA_CHECK(cudaFree(*p));
  *p = nullptr;
  *cap = 0;
  const size_t want = bytes + bytes / 8 + 256;
  const cudaError_t e = cudaMalloc(p, want);
  if (e != cudaSuccess) {
    set_error("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
    return SAI_E_NOMEM;
  }
  *cap = want;
  return SAI_OK;
}

int format_scores(FormatState& f, const sai_format_input* in, cudaStream_t st, int64_t* sizes) {
  SAI_REQUIRE(sizes, "sai_engine_format_scores: NULL sizes");
  bool has_u, has_q;
  if (int rc = check_input(in, &has_u, &has_q)) return rc;
  const int64_t nb = in->n_blocks, n = in->n_rows;
  const int64_t nu = has_u ? in->n_u_cand : 0, nq = has_q ? in->n_q_cand : 0;
  f.timed = false;
  for (int k = 0; k < 3; ++k) f.size[k] = sizes[k] = 0;
  if (n == 0) return SAI_OK;
  if (!f.ev[0])
    for (auto& ev : f.ev) SAI_CUDA_CHECK(cudaEventCreate(&ev));

  // inputs: one grow-only device buffer, one copy per column
  struct Col {
    const void* host;
    size_t bytes;
    size_t at;
  };
  Col cols[] = {
      {in->block_rows, sizeof(int64_t) * (nb + 1), 0}, {in->block_str, sizeof(int64_t) * 4 * nb, 0},
      {in->strings, (size_t)in->strings_len, 0},         {in->start, sizeof(int64_t) * n, 0},
      {in->end, sizeof(int64_t) * n, 0},                 {in->nsnps, sizeof(int32_t) * n, 0},
      {has_u ? in->u : nullptr, has_u ? sizeof(int64_t) * n : 0, 0},
      {has_u ? in->u_start : nullptr, has_u ? sizeof(int64_t) * n : 0, 0},
      {has_q ? in->q : nullptr, has_q ? sizeof(double) * n : 0, 0},
      {has_q ? in->q_start : nullptr, has_q ? sizeof(int64_t) * n : 0, 0},
      {has_q ? in->q_cnt : nullptr, has_q ? sizeof(int32_t) * n : 0, 0},
      {in->u_cand, sizeof(int32_t) * nu, 0},             {in->q_cand, sizeof(int32_t) * nq, 0},
      {in->field, sizeof(int32_t) * in->n_fields, 0},    {in->vals, sizeof(double) * n * in->n_vals, 0},
  };
  size_t total = 0;
  for (auto& c : cols) c.at = total, total += align256(c.bytes);
  if (int rc = grow_dev(&f.in, &f.in_cap, total + 256)) return rc;
  char* base = static_cast<char*>(f.in);
  SAI_CUDA_CHECK(cudaEventRecord(f.ev[0], st));
  for (const auto& c : cols)
    if (c.bytes) SAI_CUDA_CHECK(cudaMemcpyAsync(base + c.at, c.host, c.bytes, cudaMemcpyHostToDevice, st));
  SAI_CUDA_CHECK(cudaEventRecord(f.ev[1], st));
  auto dev = [&](int i) { return base + cols[i].at; };

  // scratch: three length arrays [n + 1], the candidates' digit scans [nu + 1], [nq + 1], scan chunks
  const int64_t n_chunk = (std::max(std::max(n, nu), nq) + 1023) / 1024 + 1;
  const size_t lens_at = 0, up_at = lens_at + align256(sizeof(int64_t) * 3 * (n + 1));
  const size_t qp_at = up_at + align256(sizeof(int64_t) * (nu + 1));
  const size_t ch_at = qp_at + align256(sizeof(int64_t) * (nq + 1));
  void* scratch = nullptr;
  if (int rc = scratch_alloc(&scratch, ch_at + sizeof(int64_t) * n_chunk, st)) return rc;
  char* sb = static_cast<char*>(scratch);
  int64_t* lens = reinterpret_cast<int64_t*>(sb + lens_at);
  int64_t* u_pref = reinterpret_cast<int64_t*>(sb + up_at);
  int64_t* q_pref = reinterpret_cast<int64_t*>(sb + qp_at);
  int64_t* chunk = reinterpret_cast<int64_t*>(sb + ch_at);

  FmtArgs a{};
  a.n_blocks = nb;
  a.n_rows = n;
  a.block_rows = reinterpret_cast<const int64_t*>(dev(0));
  a.block_str = reinterpret_cast<const int64_t*>(dev(1));
  a.strings = dev(2);
  a.start = reinterpret_cast<const int64_t*>(dev(3));
  a.end = reinterpret_cast<const int64_t*>(dev(4));
  a.nsnps = reinterpret_cast<const int32_t*>(dev(5));
  a.u = reinterpret_cast<const int64_t*>(dev(6));
  a.u_start = reinterpret_cast<const int64_t*>(dev(7));
  a.q = reinterpret_cast<const double*>(dev(8));
  a.q_start = reinterpret_cast<const int64_t*>(dev(9));
  a.q_cnt = reinterpret_cast<const int32_t*>(dev(10));
  a.u_cand = reinterpret_cast<const int32_t*>(dev(11));
  a.q_cand = reinterpret_cast<const int32_t*>(dev(12));
  a.field = reinterpret_cast<const int32_t*>(dev(13));
  a.vals = reinterpret_cast<const double*>(dev(14));
  a.n_fields = in->n_fields;
  a.n_vals = in->n_vals;
  a.u_pref = u_pref;
  a.q_pref = q_pref;

  // length pass + scan
  const int rows_grid = grid_for(n, 256);
  if (has_u) {
    if (nu) k_cand_digits<<<grid_for(nu, 256), 256, 0, st>>>(a.u_cand, nu, u_pref);
    scan_lengths(u_pref, nu, chunk, st);
  }
  if (has_q) {
    if (nq) k_cand_digits<<<grid_for(nq, 256), 256, 0, st>>>(a.q_cand, nq, q_pref);
    scan_lengths(q_pref, nq, chunk, st);
  }
  int64_t* len[3] = {lens, lens + (n + 1), lens + 2 * (n + 1)};
  k_row_len<<<rows_grid, 256, 0, st>>>(a, len[0]);
  scan_lengths(len[0], n, chunk, st);
  if (has_u) {
    k_log_len<true><<<rows_grid, 256, 0, st>>>(a, len[1]);
    scan_lengths(len[1], n, chunk, st);
  }
  if (has_q) {
    k_log_len<false><<<rows_grid, 256, 0, st>>>(a, len[2]);
    scan_lengths(len[2], n, chunk, st);
  }
  SAI_CUDA_CHECK(cudaGetLastError());
  SAI_CUDA_CHECK(cudaEventRecord(f.ev[2], st));
  const bool want[3] = {true, has_u, has_q};
  for (int k = 0; k < 3; ++k)
    if (want[k]) SAI_CUDA_CHECK(cudaMemcpyAsync(&f.size[k], len[k] + n, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  SAI_CUDA_CHECK(cudaStreamSynchronize(st));

  // write pass into texts of exactly the scanned sizes
  for (int k = 0; k < 3; ++k)
    if (int rc = grow_dev(reinterpret_cast<void**>(&f.text[k]), &f.text_cap[k], (size_t)f.size[k] + 256)) return rc;
  SAI_CUDA_CHECK(cudaEventRecord(f.ev[3], st));
  k_row_write<<<rows_grid, 256, 0, st>>>(a, len[0], f.text[0]);
  const int warp_grid = grid_for(n * 32, 256);
  if (has_u) k_log_write<true><<<warp_grid, 256, 0, st>>>(a, len[1], f.text[1]);
  if (has_q) k_log_write<false><<<warp_grid, 256, 0, st>>>(a, len[2], f.text[2]);
  SAI_CUDA_CHECK(cudaGetLastError());
  SAI_CUDA_CHECK(cudaEventRecord(f.ev[4], st));
  if (int rc = scratch_free(scratch, st)) return rc;
  f.timed = true;
  for (int k = 0; k < 3; ++k) sizes[k] = f.size[k];
  return SAI_OK;
}

int format_text(FormatState& f, int which, char* out, int64_t cap, cudaStream_t st) {
  SAI_REQUIRE(which >= 0 && which < 3, "sai_engine_format_text: text %d (0..2)", which);
  SAI_REQUIRE(cap >= f.size[which], "sai_engine_format_text: %lld bytes do not hold the %lld of text %d",
              (long long)cap, (long long)f.size[which], which);
  SAI_REQUIRE(out || f.size[which] == 0, "sai_engine_format_text: NULL output");
  if (f.size[which])
    SAI_CUDA_CHECK(cudaMemcpyAsync(out, f.text[which], (size_t)f.size[which], cudaMemcpyDeviceToHost, st));
  SAI_CUDA_CHECK(cudaStreamSynchronize(st));
  return SAI_OK;
}

int format_stats(FormatState& f, double* out, int n) {
  SAI_REQUIRE(out && n >= 3, "sai_engine_format_stats: needs 3 values");
  for (int k = 0; k < 3; ++k) out[k] = 0;
  if (!f.timed) return SAI_OK;
  SAI_CUDA_CHECK(cudaEventSynchronize(f.ev[4]));
  float ms[3];
  SAI_CUDA_CHECK(cudaEventElapsedTime(&ms[0], f.ev[0], f.ev[1]));
  SAI_CUDA_CHECK(cudaEventElapsedTime(&ms[1], f.ev[1], f.ev[2]));
  SAI_CUDA_CHECK(cudaEventElapsedTime(&ms[2], f.ev[3], f.ev[4]));
  for (int k = 0; k < 3; ++k) out[k] = 1e-3 * ms[k];
  return SAI_OK;
}

int format_doubles_device(const double* x, int64_t n, char* out, cudaStream_t st) {
  SAI_REQUIRE(n >= 0 && (n == 0 || (x && out)), "sai_engine_format_doubles: NULL argument");
  if (n == 0) return SAI_OK;
  void* d = nullptr;
  if (int rc = scratch_alloc(&d, sizeof(double) * n + 32 * (size_t)n + 256, st)) return rc;
  double* dx = static_cast<double*>(d);
  char* dout = reinterpret_cast<char*>(dx + n);
  SAI_CUDA_CHECK(cudaMemcpyAsync(dx, x, sizeof(double) * n, cudaMemcpyHostToDevice, st));
  k_format_doubles<<<grid_for(n, 256), 256, 0, st>>>(dx, n, dout);
  SAI_CUDA_CHECK(cudaGetLastError());
  SAI_CUDA_CHECK(cudaMemcpyAsync(out, dout, 32 * (size_t)n, cudaMemcpyDeviceToHost, st));
  if (int rc = scratch_free(d, st)) return rc;
  SAI_CUDA_CHECK(cudaStreamSynchronize(st));
  return SAI_OK;
}

void format_release(FormatState& f) {
  if (f.in) cudaFree(f.in);
  for (auto* t : f.text)
    if (t) cudaFree(t);
  for (auto ev : f.ev)
    if (ev) cudaEventDestroy(ev);
  f = FormatState{};
}

}  // namespace sai

extern "C" int32_t sai_format_double(double x, char* out) {
  if (!out) return 0;
  return sai::fmt::format_double(x, out);
}

extern "C" int sai_format_doubles(const double* x, int64_t n, char* out) {
  SAI_REQUIRE(n >= 0 && (n == 0 || (x && out)), "sai_format_doubles: NULL argument");
  for (int64_t i = 0; i < n; ++i) {
    char* o = out + 32 * i;
    memset(o, 0, 32);
    sai::fmt::format_double(x[i], o);
  }
  return SAI_OK;
}
