// Outlier tables from a score file in HBM (outlier(..., text="device")); see the table block of
// include/sai_b200.h for the calls and what each leaves resident.
//
// load: the file is copied once; its newlines are counted per 16 KiB chunk, scanned and written
// as line offsets; one warp per line finds the tabs with a ballot, keeps every cell's offset within
// its line and ORs the cells' classes (parse_double.cuh) per column and pandas parse chunk.
// parse: one thread per row writes the metric columns' float64 values ([column][row], what
// sai_column_quantiles reads), Start / End, the flag "Chrom differs from the row before" (scanned
// into run numbers) and the length of the row as the outlier table prints it.
// order: a stable LSD radix sort of the rows on (chromosome rank, Start, End), 8-bit digits, digits
// that no row changes skipped.
// build: one length per (table, sorted row) -- the header for position 0 of each table, the row's
// length where the column keeps it, else 0 -- scanned once, so all tables are laid out in one
// buffer; a write pass fills it.
#include <math.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"
#include "format_double.cuh"
#include "format_kernels.cuh"
#include "parse_double.cuh"
#include "scratch.cuh"
#include "table_kernels.cuh"

namespace sai {
namespace {

constexpr int kMaxCols = SAI_TABLE_MAX_COLS;
constexpr int64_t kChunkBytes = 16384;  // 1024 threads x 16 bytes

enum : uint32_t {
  kQuoteCr = SAI_TABLE_QUOTE_CR,
  kHighByte = SAI_TABLE_HIGH_BYTE,
  kBlank = SAI_TABLE_BLANK_LINE,
  kRagged = SAI_TABLE_RAGGED,
  kLong = SAI_TABLE_LONG_LINE,
};

struct TabArgs {
  const char* text;
  const int64_t* line;  // line[r + 1] .. line[r + 2] - 1: data row r without its '\n'
  uint16_t* cell;
  int64_t n_rows, chunk_rows;
  int32_t n_cols;
  int32_t first_metric, n_metric, chrom, start, end;
  int8_t kind[kMaxCols];  // SAI_TABLE_TEXT / _INT / _FLOAT
};

// ---- load ------------------------------------------------------------------------------------------
__device__ inline int newlines16(const uint4& v, uint32_t* flags, uint32_t* pos_mask) {
  const unsigned char* b = reinterpret_cast<const unsigned char*>(&v);
  int n = 0;
  uint32_t f = 0, m = 0;
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const unsigned char c = b[i];
    if (c == '\n') ++n, m |= 1u << i;
    if (c == '\r' || c == '"') f |= kQuoteCr;
    if (c >= 0x80) f |= kHighByte;
  }
  *flags |= f;
  *pos_mask = m;
  return n;
}

__global__ void __launch_bounds__(1024) k_lines_count(const uint4* __restrict__ text, int64_t n_chunks, int64_t* cnt,
                                                      uint32_t* flags) {
  uint32_t f = 0;
  for (int64_t c = blockIdx.x; c < n_chunks; c += gridDim.x) {
    uint32_t m;
    const int k = newlines16(text[c * 1024 + threadIdx.x], &f, &m);
    int64_t total;
    block_excl_scan64(k, &total);
    if (threadIdx.x == 0) cnt[c] = total;
  }
  f = __reduce_or_sync(0xffffffffu, f);
  if ((threadIdx.x & 31) == 0 && f) atomicOr(flags, f);
}

// line[1 + k] = one past the k-th '\n'
__global__ void __launch_bounds__(1024) k_lines_write(const uint4* __restrict__ text, int64_t n_chunks,
                                                      const int64_t* __restrict__ chunk_off, int64_t* line) {
  for (int64_t c = blockIdx.x; c < n_chunks; c += gridDim.x) {
    uint32_t f = 0, m;
    const int k = newlines16(text[c * 1024 + threadIdx.x], &f, &m);
    int64_t total;
    int64_t at = chunk_off[c] + block_excl_scan64(k, &total);
    const int64_t pos = (c * 1024 + threadIdx.x) * 16;
    for (; m; m &= m - 1) line[1 + at++] = pos + __ffs(m);
  }
}

__device__ inline void cell_span(const TabArgs& a, int64_t r, int c, const char** p, int* n) {
  const int64_t s = a.line[r + 1];
  const uint16_t* off = a.cell + r * a.n_cols;
  const int64_t cs = s + off[c];
  const int64_t ce = c + 1 < a.n_cols ? s + off[c + 1] - 1 : a.line[r + 2] - 1;
  *p = a.text + cs;
  *n = (int)(ce - cs);
}

// One warp per line over a contiguous range of rows, so that a warp's class masks change parse
// chunk rarely: lane j keeps the masks of columns j, j + 32, ...
__global__ void __launch_bounds__(256) k_fields(TabArgs a, uint32_t* cls, uint32_t* flags) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t per = (a.n_rows + n_warps - 1) / n_warps;
  const int64_t r0 = warp * per, r1 = min(r0 + per, a.n_rows);
  uint32_t acc[kMaxCols / 32] = {};
  uint32_t fl = 0;
  int64_t chunk = r0 / a.chunk_rows;
  auto flush = [&]() {
#pragma unroll
    for (int j = 0; j < kMaxCols / 32; ++j) {
      const int k = lane + 32 * j;
      if (k < a.n_cols && acc[j]) atomicOr(&cls[chunk * a.n_cols + k], acc[j]);
      acc[j] = 0;
    }
  };
  for (int64_t r = r0; r < r1; ++r) {
    if (r / a.chunk_rows != chunk) {
      flush();
      chunk = r / a.chunk_rows;
    }
    const int64_t s = a.line[r + 1], e = a.line[r + 2] - 1;
    if (e == s) {
      fl |= kBlank;
      continue;
    }
    if (e - s > 65535) {
      fl |= kLong;
      continue;
    }
    uint16_t* off = a.cell + r * a.n_cols;
    if (lane == 0) off[0] = 0;
    int tabs = 0;
    for (int64_t b = s; b < e; b += 32) {
      const int64_t p = b + lane;
      const bool tab = p < e && a.text[p] == '\t';
      const unsigned m = __ballot_sync(0xffffffffu, tab);
      if (tab) {
        const int k = tabs + __popc(m & ((1u << lane) - 1)) + 1;
        if (k < a.n_cols) off[k] = (uint16_t)(p + 1 - s);
      }
      tabs += __popc(m);
    }
    if (tabs != a.n_cols - 1) {
      fl |= kRagged;
      continue;
    }
    __syncwarp();
#pragma unroll
    for (int j = 0; j < kMaxCols / 32; ++j) {
      const int k = lane + 32 * j;
      if (k < a.n_cols) {
        const char* p;
        int n;
        cell_span(a, r, k, &p, &n);
        acc[j] |= parse::classify_cell(p, n);
      }
    }
    __syncwarp();
  }
  if (r0 < r1) flush();
  if (lane == 0 && fl) atomicOr(flags, fl);
}

// ---- parse -----------------------------------------------------------------------------------------
__device__ inline double cell_double(int kind, const char* p, int n) {
  if (kind == SAI_TABLE_INT) {
    int64_t v = 0;
    parse::parse_int64(p, n, &v);
    return (double)v;
  }
  if (parse::is_na(p, n)) return __longlong_as_double(0x7ff8000000000000ll);
  return parse::float_cell(p, n);
}

__device__ inline int64_t cell_int(const TabArgs& a, int64_t r, int c) {
  const char* p;
  int n;
  cell_span(a, r, c, &p, &n);
  int64_t v = 0;
  parse::parse_int64(p, n, &v);
  return v;
}

// Appends to o (or only counts, o == nullptr).
struct Out {
  char* o;
  int64_t n = 0;
  __device__ void put(const char* s, int64_t len) {
    if (o)
      for (int64_t i = 0; i < len; ++i) o[n + i] = s[i];
    n += len;
  }
  __device__ void ch(char c) {
    if (o) o[n] = c;
    ++n;
  }
};

// a data row as ScoreTable.format_cell prints it: int64 in decimal, float64 as repr ("nan" for NA),
// text as its bytes ("nan" for NA)
__device__ int64_t row_text(const TabArgs& a, int64_t r, char* out) {
  Out t{out};
  for (int c = 0; c < a.n_cols; ++c) {
    if (c) t.ch('\t');
    const char* p;
    int n;
    cell_span(a, r, c, &p, &n);
    const int kind = a.kind[c];
    char buf[fmt::kMaxDoubleChars];
    if (kind == SAI_TABLE_INT) {
      int64_t v = 0;
      parse::parse_int64(p, n, &v);
      t.put(buf, fmt::format_int64(v, buf));
    } else if (parse::is_na(p, n)) {
      t.put("nan", 3);
    } else if (kind == SAI_TABLE_FLOAT) {
      t.put(buf, fmt::format_double(parse::float_cell(p, n), buf));
    } else {
      t.put(p, n);
    }
  }
  t.ch('\n');
  return t.n;
}

__device__ inline bool same_cell(const TabArgs& a, int64_t r, int64_t q, int c) {
  const char *p, *s;
  int n, m;
  cell_span(a, r, c, &p, &n);
  cell_span(a, q, c, &s, &m);
  if (n != m) return false;
  for (int i = 0; i < n; ++i)
    if (p[i] != s[i]) return false;
  return true;
}

struct RowCols {
  double* vals;         // [n_metric][n_rows]
  unsigned* first;      // [n_metric]: first row with a value
  int64_t* run;         // [n_rows + 1]: 1 where Chrom differs from the row before, scanned later
  int64_t* row_len;     // [n_rows]
  int64_t *start, *end; // [n_rows]
};

// a warp takes 32 consecutive rows, so that the first row with a value is one warp minimum
__global__ void __launch_bounds__(256) k_values(TabArgs a, RowCols o) {
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t r0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) - lane; r0 < a.n_rows; r0 += stride) {
    const int64_t r = r0 + lane;
    const bool live = r < a.n_rows;
    for (int m = 0; m < a.n_metric; ++m) {
      double v = 0. / 0.;
      if (live) {
        const char* p;
        int n;
        cell_span(a, r, a.first_metric + m, &p, &n);
        v = cell_double(a.kind[a.first_metric + m], p, n);
        o.vals[m * a.n_rows + r] = v;
      }
      const unsigned mn = __reduce_min_sync(0xffffffffu, live && v == v ? (unsigned)r : 0xffffffffu);
      if (lane == 0 && mn != 0xffffffffu) atomicMin(&o.first[m], mn);
    }
    if (!live) continue;
    o.start[r] = cell_int(a, r, a.start);
    o.end[r] = cell_int(a, r, a.end);
    o.run[r] = r == 0 || !same_cell(a, r, r - 1, a.chrom);
    o.row_len[r] = row_text(a, r, nullptr);
  }
}

// run[] scanned: a run starts at r where run[r + 1] != run[r]; its name is r's Chrom cell
__global__ void k_run_heads(TabArgs a, const int64_t* __restrict__ run, int64_t* head_off, int64_t* head_len) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < a.n_rows; r += (int64_t)gridDim.x * blockDim.x)
    if (run[r + 1] != run[r]) {
      const char* p;
      int n;
      cell_span(a, r, a.chrom, &p, &n);
      head_off[run[r]] = p - a.text;
      head_len[run[r]] = n;
    }
}

__global__ void k_first_values(const double* vals, const unsigned* first, int n_metric, int64_t n_rows, double* out) {
  const int m = threadIdx.x;
  if (m < n_metric) out[m] = first[m] < n_rows ? vals[m * n_rows + first[m]] : __longlong_as_double(0x7ff8000000000000ll);
}

// ---- order -----------------------------------------------------------------------------------------
__device__ inline uint64_t flip(int64_t v) { return (uint64_t)v ^ 0x8000000000000000ull; }

// keys[0] = chromosome rank, keys[1] = Start, keys[2] = End (order-preserving unsigned); mask[2k] |=,
// mask[2k + 1] &= every key, so that a digit no row changes is skipped
__global__ void k_sort_keys(int64_t n, const int64_t* __restrict__ run, const int32_t* __restrict__ run_rank,
                            const int64_t* __restrict__ start, const int64_t* __restrict__ end, uint64_t* keys,
                            int32_t* perm, unsigned long long* mask) {
  unsigned long long o[3] = {0, 0, 0}, d[3] = {~0ull, ~0ull, ~0ull};
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
    const uint64_t k[3] = {(uint64_t)run_rank[run[r + 1] - 1], flip(start[r]), flip(end[r])};
    for (int j = 0; j < 3; ++j) {
      keys[j * n + r] = k[j];
      o[j] |= k[j];
      d[j] &= k[j];
    }
    perm[r] = (int32_t)r;
  }
  for (int j = 0; j < 3; ++j) {
    for (int s = 16; s > 0; s >>= 1) {
      o[j] |= __shfl_xor_sync(0xffffffffu, o[j], s);
      d[j] &= __shfl_xor_sync(0xffffffffu, d[j], s);
    }
    if ((threadIdx.x & 31) == 0) {
      atomicOr(&mask[2 * j], o[j]);
      atomicAnd(&mask[2 * j + 1], d[j]);
    }
  }
}

constexpr int kRadixTile = 256;  // rows per radix tile = threads per block

__global__ void __launch_bounds__(kRadixTile) k_radix_count(const int32_t* __restrict__ perm, const uint64_t* __restrict__ key,
                                                       int shift, int64_t n, int64_t n_tiles, int64_t* hist) {
  __shared__ int cnt[256];
  for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    cnt[threadIdx.x] = 0;
    __syncthreads();
    const int64_t i = t * kRadixTile + threadIdx.x;
    if (i < n) atomicAdd(&cnt[(key[perm[i]] >> shift) & 255], 1);
    __syncthreads();
    hist[threadIdx.x * n_tiles + t] = cnt[threadIdx.x];  // digit-major: the scan orders digits, then tiles
    __syncthreads();
  }
}

// stable: within a tile, rows of one digit keep their order (warp match + counts per warp)
__global__ void __launch_bounds__(kRadixTile) k_radix_scatter(const int32_t* __restrict__ perm, const uint64_t* __restrict__ key,
                                                         int shift, int64_t n, int64_t n_tiles,
                                                         const int64_t* __restrict__ off, int32_t* out) {
  __shared__ int wcnt[kRadixTile / 32][256];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    for (int j = threadIdx.x; j < (kRadixTile / 32) * 256; j += kRadixTile) (&wcnt[0][0])[j] = 0;
    __syncthreads();
    const int64_t i = t * kRadixTile + threadIdx.x;
    const bool live = i < n;
    const int32_t row = live ? perm[i] : 0;
    const int d = live ? (int)((key[row] >> shift) & 255) : 256;
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    const int before = __popc(peers & ((1u << lane) - 1));
    if (live && before == 0) wcnt[w][d] = __popc(peers);
    __syncthreads();
    int run = 0;
    for (int ww = 0; ww < kRadixTile / 32; ++ww) {
      const int c = wcnt[ww][threadIdx.x];
      wcnt[ww][threadIdx.x] = run;
      run += c;
    }
    __syncthreads();
    if (live) out[off[(int64_t)d * n_tiles + t] + wcnt[w][d] + before] = row;
    __syncthreads();
  }
}

// ---- build -----------------------------------------------------------------------------------------
struct BuildArgs {
  int32_t n_tables;
  int64_t header_len;
  const int32_t* perm;
  const int64_t* row_len;
  const double* vals;
  double thr[kMaxCols];
  int8_t strict[kMaxCols];  // '>' (columns named U...) rather than '>='
};

__global__ void k_table_len(BuildArgs b, int64_t n, int64_t* lens) {
  const int64_t total = (int64_t)b.n_tables * (n + 1);
  for (int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; x < total; x += (int64_t)gridDim.x * blockDim.x) {
    const int m = (int)(x / (n + 1));
    const int64_t i = x - m * (n + 1);
    if (i == 0) {
      lens[x] = b.header_len;
      continue;
    }
    const int32_t row = b.perm[i - 1];
    const double v = b.vals[m * n + row], thr = b.thr[m];
    lens[x] = (b.strict[m] ? v > thr : v >= thr) ? b.row_len[row] : 0;  // NaN is never kept
  }
}

__global__ void k_table_offsets(const int64_t* lens, int32_t n_tables, int64_t n, int64_t* offs) {
  const int m = threadIdx.x;
  if (m <= n_tables) offs[m] = lens[(int64_t)m * (n + 1)];
}

__global__ void k_table_write(TabArgs a, BuildArgs b, const int64_t* __restrict__ lens, char* out) {
  const int64_t n = a.n_rows, total = (int64_t)b.n_tables * (n + 1);
  for (int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; x < total; x += (int64_t)gridDim.x * blockDim.x) {
    const int64_t at = lens[x];
    if (lens[x + 1] == at) continue;
    const int64_t i = x % (n + 1);
    if (i == 0) {
      for (int64_t k = 0; k < b.header_len; ++k) out[at + k] = a.text[k];
    } else {
      row_text(a, b.perm[i - 1], out + at);
    }
  }
}

__global__ void k_parse_doubles(const char* text, const int64_t* offs, int64_t n, double* out, uint8_t* ok) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    ok[i] = parse::xstrtod(text + offs[i], (int)(offs[i + 1] - offs[i]), &out[i]);
}

int grow(DevBuf& b, size_t bytes) { return grow_dev(&b.p, &b.cap, bytes); }

template <typename T>
T* at(DevBuf& b, size_t off_bytes = 0) {
  return reinterpret_cast<T*>(static_cast<char*>(b.p) + off_bytes);
}

// misc buffer: flags | first[kMaxCols] | first values | key masks | offsets | chunk counts ...
constexpr size_t kMiscFirst = 256, kMiscFirstVal = kMiscFirst + 4 * kMaxCols, kMiscMask = kMiscFirstVal + 8 * kMaxCols,
                 kMiscOffs = kMiscMask + 64, kMiscEnd = kMiscOffs + 8 * (kMaxCols + 1);

size_t al(size_t x) { return (x + 255) & ~size_t(255); }

TabArgs args(TableState& t) {
  TabArgs a{};
  a.text = at<char>(t.text);
  a.line = at<int64_t>(t.line);
  a.cell = at<uint16_t>(t.cell);
  a.n_rows = t.n_rows;
  a.chunk_rows = t.chunk_rows;
  a.n_cols = (int32_t)t.n_cols;
  a.first_metric = t.first_metric;
  a.n_metric = (int32_t)t.n_cols - t.first_metric;
  a.chrom = t.chrom;
  a.start = t.start;
  a.end = t.end;
  for (int c = 0; c < t.n_cols; ++c) a.kind[c] = (int8_t)t.kind[c];
  return a;
}

// rows buffer: run [n + 1] | row_len | start | end | head_off | head_len
int64_t* rows_at(TableState& t, int k) { return at<int64_t>(t.rows) + (k == 0 ? 0 : (t.n_rows + 1) + (k - 1) * t.n_rows); }

int ensure_events(TableState& t) {
  if (!t.ev[0])
    for (auto& ev : t.ev) SAI_CUDA_CHECK(cudaEventCreate(&ev));
  return SAI_OK;
}

}  // namespace

int table_load(TableState& t, const char* text, int64_t n_bytes, int32_t n_cols, int64_t chunk_rows, int64_t* info,
               cudaStream_t st) {
  SAI_REQUIRE(text && info && n_bytes > 0, "sai_engine_table_load: NULL or empty text");
  SAI_REQUIRE(n_cols >= 1 && n_cols <= kMaxCols, "sai_engine_table_load: %d columns (1..%d)", n_cols, kMaxCols);
  SAI_REQUIRE(chunk_rows >= 1, "sai_engine_table_load: chunk_rows %lld", (long long)chunk_rows);
  t.parsed = t.ordered = false;
  t.out_size = t.n_rows = t.n_chunks = 0;
  for (bool& b : t.timed) b = false;
  if (int rc = ensure_events(t)) return rc;
  const int64_t n_chunks16 = (n_bytes + kChunkBytes - 1) / kChunkBytes;
  const size_t padded = (size_t)n_chunks16 * kChunkBytes;
  if (int rc = grow(t.text, padded)) return rc;
  if (int rc = grow(t.misc, kMiscEnd + 8 * (size_t)(n_chunks16 + 1) + 8 * (size_t)((n_chunks16 + 1023) / 1024 + 2)))
    return rc;
  t.n_bytes = n_bytes;
  t.n_cols = n_cols;
  t.chunk_rows = chunk_rows;
  SAI_CUDA_CHECK(cudaEventRecord(t.ev[0], st));
  SAI_CUDA_CHECK(cudaMemcpyAsync(t.text.p, text, (size_t)n_bytes, cudaMemcpyHostToDevice, st));
  SAI_CUDA_CHECK(cudaMemsetAsync(at<char>(t.text, n_bytes), 0, padded - (size_t)n_bytes, st));
  SAI_CUDA_CHECK(cudaEventRecord(t.ev[1], st));
  t.timed[0] = true;

  uint32_t* flags = at<uint32_t>(t.misc);
  int64_t* cnt = at<int64_t>(t.misc, kMiscEnd);
  int64_t* scan_chunk = cnt + n_chunks16 + 1;
  SAI_CUDA_CHECK(cudaMemsetAsync(flags, 0, sizeof(uint32_t), st));
  const uint4* t16 = at<const uint4>(t.text);
  const int g = grid_for(n_chunks16, 1);
  k_lines_count<<<g, 1024, 0, st>>>(t16, n_chunks16, cnt, flags);
  scan_lengths(cnt, n_chunks16, scan_chunk, st);
  int64_t n_nl = 0;
  SAI_CUDA_CHECK(cudaMemcpyAsync(&n_nl, cnt + n_chunks16, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  SAI_CUDA_CHECK(cudaStreamSynchronize(st));
  const bool open_end = text[n_bytes - 1] != '\n';
  const int64_t n_lines = n_nl + (open_end ? 1 : 0);
  t.n_rows = n_lines - 1;
  SAI_REQUIRE(t.n_rows < (1ll << 31) - 1, "sai_engine_table_load: %lld rows (at most 2^31 - 2)", (long long)t.n_rows);
  t.n_chunks = t.n_rows > 0 ? (t.n_rows + chunk_rows - 1) / chunk_rows : 0;
  if (t.n_rows > 0) {
    if (int rc = grow(t.line, 8 * (size_t)(n_lines + 1))) return rc;
    if (int rc = grow(t.cell, 2 * (size_t)t.n_rows * n_cols)) return rc;
    if (int rc = grow(t.cls, 4 * (size_t)t.n_chunks * n_cols)) return rc;
    int64_t* line = at<int64_t>(t.line);
    SAI_CUDA_CHECK(cudaMemsetAsync(line, 0, sizeof(int64_t), st));
    k_lines_write<<<g, 1024, 0, st>>>(t16, n_chunks16, cnt, line);
    if (open_end) {  // the last line ends at the end of the file
      const int64_t past_end = n_bytes + 1;  // pageable: copied before the call returns
      SAI_CUDA_CHECK(cudaMemcpyAsync(line + n_lines, &past_end, sizeof(int64_t), cudaMemcpyHostToDevice, st));
    }
    SAI_CUDA_CHECK(cudaMemsetAsync(t.cls.p, 0, 4 * (size_t)t.n_chunks * n_cols, st));
    TabArgs a = args(t);
    k_fields<<<grid_for(t.n_rows * 32, 256), 256, 0, st>>>(a, at<uint32_t>(t.cls), flags);
    SAI_CUDA_CHECK(cudaGetLastError());
  }
  SAI_CUDA_CHECK(cudaEventRecord(t.ev[3], st));
  uint32_t f = 0;
  SAI_CUDA_CHECK(cudaMemcpyAsync(&f, flags, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  SAI_CUDA_CHECK(cudaStreamSynchronize(st));
  t.timed[1] = true;
  info[0] = t.n_rows;
  info[1] = t.n_chunks;
  info[2] = f;
  return SAI_OK;
}

int table_classes(TableState& t, uint32_t* out, int64_t cap, cudaStream_t st) {
  const int64_t n = t.n_chunks * t.n_cols;
  SAI_REQUIRE(out || n == 0, "sai_engine_table_classes: NULL output");
  SAI_REQUIRE(cap >= n, "sai_engine_table_classes: %lld entries do not hold %lld", (long long)cap, (long long)n);
  if (n) SAI_CUDA_CHECK(cudaMemcpyAsync(out, t.cls.p, 4 * (size_t)n, cudaMemcpyDeviceToHost, st));
  SAI_CUDA_CHECK(cudaStreamSynchronize(st));
  return SAI_OK;
}

int table_parse(TableState& t, const int32_t* kinds, int32_t first_metric, int32_t chrom, int32_t start, int32_t end,
                double* d_vals, double* first_val, int64_t* n_runs, cudaStream_t st) {
  SAI_REQUIRE(t.n_rows > 0, "sai_engine_table_parse: no table loaded");
  SAI_REQUIRE(kinds && d_vals && first_val && n_runs, "sai_engine_table_parse: NULL argument");
  SAI_REQUIRE(first_metric >= 0 && first_metric < t.n_cols, "sai_engine_table_parse: first metric column %d", first_metric);
  const int32_t cols[3] = {chrom, start, end};
  for (int32_t c : cols) SAI_REQUIRE(c >= 0 && c < t.n_cols, "sai_engine_table_parse: column %d of %lld", c, (long long)t.n_cols);
  for (int c = 0; c < t.n_cols; ++c) {
    SAI_REQUIRE(kinds[c] >= SAI_TABLE_TEXT && kinds[c] <= SAI_TABLE_FLOAT, "sai_engine_table_parse: kind %d", kinds[c]);
    t.kind[c] = kinds[c];
  }
  SAI_REQUIRE(kinds[start] == SAI_TABLE_INT && kinds[end] == SAI_TABLE_INT, "sai_engine_table_parse: Start / End not int64");
  for (int c = first_metric; c < t.n_cols; ++c)
    SAI_REQUIRE(kinds[c] != SAI_TABLE_TEXT, "sai_engine_table_parse: metric column %d is text", c);
  t.first_metric = first_metric;
  t.chrom = chrom;
  t.start = start;
  t.end = end;
  t.vals = d_vals;
  t.parsed = t.ordered = false;
  const int64_t n = t.n_rows;
  const int n_metric = (int)(t.n_cols - first_metric);
  if (int rc = grow(t.rows, 8 * (size_t)(6 * n + 1))) return rc;
  unsigned* first = at<unsigned>(t.misc, kMiscFirst);
  double* first_d = at<double>(t.misc, kMiscFirstVal);
  SAI_CUDA_CHECK(cudaEventRecord(t.ev[4], st));
  SAI_CUDA_CHECK(cudaMemsetAsync(first, 0xff, 4 * kMaxCols, st));
  RowCols o{d_vals, first, rows_at(t, 0), rows_at(t, 1), rows_at(t, 2), rows_at(t, 3)};
  TabArgs a = args(t);
  k_values<<<grid_for(n, 256), 256, 0, st>>>(a, o);
  int64_t* chunk = nullptr;
  if (int rc = scratch_alloc(reinterpret_cast<void**>(&chunk), 8 * (size_t)((n + 1023) / 1024 + 2), st)) return rc;
  scan_lengths(o.run, n, chunk, st);
  if (int rc = scratch_free(chunk, st)) return rc;
  k_run_heads<<<grid_for(n, 256), 256, 0, st>>>(a, o.run, rows_at(t, 4), rows_at(t, 5));
  k_first_values<<<1, kMaxCols, 0, st>>>(d_vals, first, n_metric, n, first_d);
  SAI_CUDA_CHECK(cudaGetLastError());
  SAI_CUDA_CHECK(cudaEventRecord(t.ev[5], st));
  SAI_CUDA_CHECK(cudaMemcpyAsync(first_val, first_d, 8 * (size_t)n_metric, cudaMemcpyDeviceToHost, st));
  SAI_CUDA_CHECK(cudaMemcpyAsync(&t.n_runs, o.run + n, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  SAI_CUDA_CHECK(cudaStreamSynchronize(st));
  t.timed[2] = true;
  t.parsed = true;
  *n_runs = t.n_runs;
  return SAI_OK;
}

int table_runs(TableState& t, int64_t* off, int64_t* len, int64_t cap, cudaStream_t st) {
  SAI_REQUIRE(t.parsed, "sai_engine_table_runs: no table parsed");
  SAI_REQUIRE(off && len && cap >= t.n_runs, "sai_engine_table_runs: the output does not hold %lld runs", (long long)t.n_runs);
  SAI_CUDA_CHECK(cudaMemcpyAsync(off, rows_at(t, 4), 8 * (size_t)t.n_runs, cudaMemcpyDeviceToHost, st));
  SAI_CUDA_CHECK(cudaMemcpyAsync(len, rows_at(t, 5), 8 * (size_t)t.n_runs, cudaMemcpyDeviceToHost, st));
  SAI_CUDA_CHECK(cudaStreamSynchronize(st));
  return SAI_OK;
}

// sort buffer: keys [3][n] uint64 | perm [2][n] int32 | run_rank [n] int32 | hist [256 n_tiles + 1] | scan chunks
int table_order(TableState& t, const int32_t* run_rank, int64_t n_runs, cudaStream_t st) {
  SAI_REQUIRE(t.parsed, "sai_engine_table_order: no table parsed");
  SAI_REQUIRE(run_rank && n_runs == t.n_runs, "sai_engine_table_order: %lld ranks for %lld runs", (long long)n_runs,
              (long long)t.n_runs);
  const int64_t n = t.n_rows, n_tiles = (n + kRadixTile - 1) / kRadixTile, n_hist = 256 * n_tiles;
  const size_t keys_at = 0, perm_at = keys_at + al(24 * (size_t)n), rank_at = perm_at + al(8 * (size_t)n);
  const size_t hist_at = rank_at + al(4 * (size_t)n), chunk_at = hist_at + al(8 * (size_t)(n_hist + 1));
  if (int rc = grow(t.sort, chunk_at + 8 * (size_t)((n_hist + 1023) / 1024 + 2))) return rc;
  uint64_t* keys = at<uint64_t>(t.sort, keys_at);
  int32_t* perm[2] = {at<int32_t>(t.sort, perm_at), at<int32_t>(t.sort, perm_at) + n};
  int32_t* rank = at<int32_t>(t.sort, rank_at);
  int64_t* hist = at<int64_t>(t.sort, hist_at);
  int64_t* chunk = at<int64_t>(t.sort, chunk_at);
  unsigned long long* mask = at<unsigned long long>(t.misc, kMiscMask);
  SAI_CUDA_CHECK(cudaEventRecord(t.ev[6], st));
  SAI_CUDA_CHECK(cudaMemcpyAsync(rank, run_rank, 4 * (size_t)n_runs, cudaMemcpyHostToDevice, st));
  unsigned long long m0[6] = {0, ~0ull, 0, ~0ull, 0, ~0ull};
  SAI_CUDA_CHECK(cudaMemcpyAsync(mask, m0, sizeof(m0), cudaMemcpyHostToDevice, st));
  k_sort_keys<<<grid_for(n, 256), 256, 0, st>>>(n, rows_at(t, 0), rank, rows_at(t, 2), rows_at(t, 3), keys, perm[0], mask);
  unsigned long long m[6];
  SAI_CUDA_CHECK(cudaMemcpyAsync(m, mask, sizeof(m), cudaMemcpyDeviceToHost, st));
  SAI_CUDA_CHECK(cudaStreamSynchronize(st));
  int cur = 0;
  const int g = grid_for(n_tiles, 1);
  for (int j = 2; j >= 0; --j) {  // least significant key first: End, Start, chromosome rank
    const unsigned long long varying = m[2 * j] ^ m[2 * j + 1];
    for (int shift = 0; shift < 64; shift += 8) {
      if (((varying >> shift) & 255) == 0) continue;
      k_radix_count<<<g, kRadixTile, 0, st>>>(perm[cur], keys + j * n, shift, n, n_tiles, hist);
      scan_lengths(hist, n_hist, chunk, st);
      k_radix_scatter<<<g, kRadixTile, 0, st>>>(perm[cur], keys + j * n, shift, n, n_tiles, hist, perm[cur ^ 1]);
      cur ^= 1;
    }
  }
  SAI_CUDA_CHECK(cudaGetLastError());
  if (cur == 1) SAI_CUDA_CHECK(cudaMemcpyAsync(perm[0], perm[1], 4 * (size_t)n, cudaMemcpyDeviceToDevice, st));
  SAI_CUDA_CHECK(cudaEventRecord(t.ev[7], st));
  t.timed[3] = true;
  t.ordered = true;
  return SAI_OK;
}

int table_build(TableState& t, const double* thr, const int32_t* strict, int64_t* offsets, cudaStream_t st) {
  SAI_REQUIRE(t.ordered, "sai_engine_table_build: no row order (sai_engine_table_order)");
  SAI_REQUIRE(thr && strict && offsets, "sai_engine_table_build: NULL argument");
  const int64_t n = t.n_rows;
  const int32_t T = (int32_t)(t.n_cols - t.first_metric);
  BuildArgs b{};
  b.n_tables = T;
  b.perm = at<int32_t>(t.sort, al(24 * (size_t)n));
  b.row_len = rows_at(t, 1);
  b.vals = t.vals;
  for (int m = 0; m < T; ++m) {
    b.thr[m] = thr[m];
    b.strict[m] = strict[m] != 0;
  }
  int64_t line1 = 0;
  SAI_CUDA_CHECK(cudaMemcpyAsync(&line1, at<int64_t>(t.line) + 1, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  SAI_CUDA_CHECK(cudaStreamSynchronize(st));
  b.header_len = line1;  // the header line with its '\n'
  const int64_t total = (int64_t)T * (n + 1);
  if (int rc = grow(t.lens, 8 * (size_t)(total + 1) + 8 * (size_t)((total + 1023) / 1024 + 2))) return rc;
  int64_t* lens = at<int64_t>(t.lens);
  int64_t* chunk = lens + total + 1;
  int64_t* offs = at<int64_t>(t.misc, kMiscOffs);
  SAI_CUDA_CHECK(cudaEventRecord(t.ev[8], st));
  k_table_len<<<grid_for(total, 256), 256, 0, st>>>(b, n, lens);
  scan_lengths(lens, total, chunk, st);
  k_table_offsets<<<1, kMaxCols + 1, 0, st>>>(lens, T, n, offs);
  SAI_CUDA_CHECK(cudaGetLastError());
  SAI_CUDA_CHECK(cudaMemcpyAsync(offsets, offs, 8 * (size_t)(T + 1), cudaMemcpyDeviceToHost, st));
  SAI_CUDA_CHECK(cudaStreamSynchronize(st));
  t.out_size = offsets[T];
  if (int rc = grow(t.out, (size_t)t.out_size + 256)) return rc;
  k_table_write<<<grid_for(total, 256), 256, 0, st>>>(args(t), b, lens, at<char>(t.out));
  SAI_CUDA_CHECK(cudaGetLastError());
  SAI_CUDA_CHECK(cudaEventRecord(t.ev[9], st));
  t.timed[4] = true;
  return SAI_OK;
}

int table_text(TableState& t, char* out, int64_t cap, cudaStream_t st) {
  SAI_REQUIRE(cap >= t.out_size, "sai_engine_table_text: %lld bytes do not hold %lld", (long long)cap, (long long)t.out_size);
  SAI_REQUIRE(out || t.out_size == 0, "sai_engine_table_text: NULL output");
  SAI_CUDA_CHECK(cudaEventRecord(t.ev[10], st));
  if (t.out_size) SAI_CUDA_CHECK(cudaMemcpyAsync(out, t.out.p, (size_t)t.out_size, cudaMemcpyDeviceToHost, st));
  SAI_CUDA_CHECK(cudaEventRecord(t.ev[11], st));
  SAI_CUDA_CHECK(cudaStreamSynchronize(st));
  t.timed[5] = true;
  return SAI_OK;
}

int table_stats(TableState& t, double* out, int n) {
  SAI_REQUIRE(out && n >= 6, "sai_engine_table_stats: needs 6 values");
  // copy in, tokenise + classify (ev[1] .. ev[3]), parse, sort, format, copy back
  const int from[6] = {0, 1, 4, 6, 8, 10}, to[6] = {1, 3, 5, 7, 9, 11};
  for (int k = 0; k < 6; ++k) {
    out[k] = 0;
    if (!t.timed[k]) continue;
    SAI_CUDA_CHECK(cudaEventSynchronize(t.ev[to[k]]));
    float ms = 0;
    SAI_CUDA_CHECK(cudaEventElapsedTime(&ms, t.ev[from[k]], t.ev[to[k]]));
    out[k] = 1e-3 * ms;
  }
  return SAI_OK;
}

int parse_doubles_device(const char* text, const int64_t* offs, int64_t n, double* out, uint8_t* ok, cudaStream_t st) {
  SAI_REQUIRE(n >= 0 && (n == 0 || (text && offs && out && ok)), "sai_engine_parse_doubles: NULL argument");
  if (n == 0) return SAI_OK;
  const int64_t bytes = offs[n];
  const size_t text_at = 0, offs_at = al((size_t)bytes + 1), out_at = offs_at + al(8 * (size_t)(n + 1)),
               ok_at = out_at + al(8 * (size_t)n);
  void* d = nullptr;
  if (int rc = scratch_alloc(&d, ok_at + (size_t)n, st)) return rc;
  char* base = static_cast<char*>(d);
  SAI_CUDA_CHECK(cudaMemcpyAsync(base + text_at, text, (size_t)bytes, cudaMemcpyHostToDevice, st));
  SAI_CUDA_CHECK(cudaMemcpyAsync(base + offs_at, offs, 8 * (size_t)(n + 1), cudaMemcpyHostToDevice, st));
  k_parse_doubles<<<grid_for(n, 256), 256, 0, st>>>(base + text_at, reinterpret_cast<int64_t*>(base + offs_at), n,
                                                     reinterpret_cast<double*>(base + out_at),
                                                     reinterpret_cast<uint8_t*>(base + ok_at));
  SAI_CUDA_CHECK(cudaGetLastError());
  SAI_CUDA_CHECK(cudaMemcpyAsync(out, base + out_at, 8 * (size_t)n, cudaMemcpyDeviceToHost, st));
  SAI_CUDA_CHECK(cudaMemcpyAsync(ok, base + ok_at, (size_t)n, cudaMemcpyDeviceToHost, st));
  if (int rc = scratch_free(d, st)) return rc;
  SAI_CUDA_CHECK(cudaStreamSynchronize(st));
  return SAI_OK;
}

void table_release(TableState& t) {
  for (DevBuf* b : {&t.text, &t.line, &t.cell, &t.cls, &t.misc, &t.rows, &t.sort, &t.lens, &t.out})
    if (b->p) cudaFree(b->p);
  for (auto ev : t.ev)
    if (ev) cudaEventDestroy(ev);
  t = TableState{};
}

}  // namespace sai

extern "C" int sai_parse_doubles(const char* text, const int64_t* offs, int64_t n, double* out, uint8_t* ok) {
  SAI_REQUIRE(n >= 0 && (n == 0 || (text && offs && out && ok)), "sai_parse_doubles: NULL argument");
  for (int64_t i = 0; i < n; ++i) ok[i] = sai::parse::xstrtod(text + offs[i], (int)(offs[i + 1] - offs[i]), &out[i]);
  return SAI_OK;
}

extern "C" int sai_classify_cells(const char* text, const int64_t* offs, int64_t n, uint8_t* cls) {
  SAI_REQUIRE(n >= 0 && (n == 0 || (text && offs && cls)), "sai_classify_cells: NULL argument");
  for (int64_t i = 0; i < n; ++i) cls[i] = sai::parse::classify_cell(text + offs[i], (int)(offs[i + 1] - offs[i]));
  return SAI_OK;
}
