// Device VCF genotype parser: VCF text resident in HBM -> tiled bit-planes + positions.
//
// The host parser (vcf_parse.cu: GtParser::scan / parse_record / gt_sum) is the specification; this
// file reproduces it record for record and value for value on one text slice (any run of complete
// lines) per sai_vcf_tiles_device call:
//   1. newline index: per 8 KB segment a newline count, an exclusive scan, then the line ends in
//      file order (per-thread counts, warp ballot / popc ranks, block scan);
//   2. record pass, one warp per line: empty and '#' lines skipped, a trailing '\r' stripped, the
//      first nine tabs found with ballots, then CHROM / POS / region / REF / first ALT /
//      ancestral-allele table (binary search, flip when ALT is ancestral) / GT index in FORMAT;
//      a record without a sample column (fewer than nine tabs) is dropped, as the host drops it;
//   3. site numbering: per 1024 lines a keep count, an exclusive scan that also advances the
//      device-side site counter of sai_vcf_state (slices chain without a host sync), then the
//      kept lines in file order and pos[site];
//   4. genotype pass, one warp per kept record: lane j parses individual 32g + j of every group of
//      every population into the allele sum (gt_sum semantics), one __ballot_sync per bit-plane
//      gives the plane word.  A record whose fields are all three characters wide (the regular
//      `x|y` diploid record, GT first) is addressed directly at samples + 4*col; any other record
//      first has its field offsets written to the warp's scratch row by a cooperative tab scan;
//   5. the sites behind the last one written, up to the end of its tile, are coded all-missing --
//      so after every call the tiles are exactly what sai_pack_i8_all writes for the sites so far.
#include <string.h>

#include "vcf_genome.cuh"

namespace sai {

namespace {

constexpr int kSegBytes = 8192;       // newline pass: bytes per block (256 threads x 32 bytes)
constexpr int kLinesPerChunk = 1024;  // site numbering: lines per block
constexpr int kWarpsPerBlock = 8;

struct SliceInfo {
  int32_t n_lines;
  int32_t n_kept;
  int64_t site_base;
  int32_t n_bnd;  // genome: kept records whose chromosome differs from the one before (bnd)
  int32_t n_seg;  // genome: runs of one chromosome's kept records in the slice (seg_*)
};

struct Scratch {
  SliceInfo* info;
  int32_t* seg_cnt;   // [n_seg]
  int32_t* seg_off;   // [n_seg]
  int32_t* line_end;  // [len]
  int32_t* rec_samp;  // [len] offset of the first sample field
  int32_t* rec_end;   // [len] end of the line ('\r' stripped)
  int32_t* rec_pos;   // [len]
  int32_t* rec_meta;  // [len] bit 0 keep, bit 1 flip, bits 2.. GT index
  int32_t* chunk_cnt; // [n_chunk]
  int32_t* chunk_off; // [n_chunk]
  int32_t* kept;      // line index of the slice's k-th kept record: reuses line_end, which only the record pass reads
  int32_t* fields;    // [n_geno_warps][max_column + 1] field offsets of irregular records
  // genome parse only
  int32_t* rec_chrom; // [len] chromosome of the line, -1: not listed
  uint32_t* rec_span; // [len] POS for the chromosome's span
  int32_t* bnd;       // [n_chrom + 1] slice index of a kept record that starts a run (unordered)
  int32_t* seg_k;     // [n_chrom + 2] first kept record (slice index) of run j, ascending
  int64_t* seg_site;  // [n_chrom + 2] its site
  int64_t* seg_gap;   // [n_chrom + 2] end of the run before it: [seg_gap, seg_site) are padding sites
};

// Slice scratch and session of the negative-value table (vcf_genome.cuh, VcfNegSession)
struct NegArgs {
  int32_t* cnt;        // [n_pops * n_kept + 1] missing calls of (population, kept record); then their exclusive scan
  uint32_t* at;        // [n_pops * n_kept] first entry of (population, kept record), relative to slice_base
  int2* pending;       // [n_geno_warps][row] (individual, value) of the record's population being parsed
  int32_t* chunk_cnt;  // scan of cnt: per 1024 items
  int32_t* chunk_off;
  int32_t row;         // largest population
  int32_t n_pops;
  VcfNegSession t;
};

inline size_t al(size_t x) { return (x + 255) & ~size_t(255); }

int geno_warps() { return sm_count() * 4 * kWarpsPerBlock; }

// a kept record is at least 11 bytes (CHROM, nine tabs, newline)
inline size_t max_kept(int64_t len) { return (size_t)len / 11 + 2; }

// byte size of the negative-value scratch of a slice and, when base != null, its carving
size_t carve_neg(const sai_vcf_query& q, int64_t len, char* base, NegArgs* a) {
  int32_t row = 1;
  for (int p = 0; p < q.lay.n_pops; ++p) row = row > q.lay.pop[p].n_samples ? row : q.lay.pop[p].n_samples;
  const size_t n_item = (size_t)q.lay.n_pops * max_kept(len);
  const size_t n_chunk = n_item / 1024 + 2;
  size_t at = 0;
  auto take = [&](size_t bytes) {
    char* p = base ? base + at : nullptr;
    at += al(bytes);
    return p;
  };
  NegArgs t{};
  t.cnt = reinterpret_cast<int32_t*>(take(4 * (n_item + 1)));
  t.at = reinterpret_cast<uint32_t*>(take(4 * n_item));
  t.pending = reinterpret_cast<int2*>(take(8 * (size_t)geno_warps() * (size_t)row));
  t.chunk_cnt = reinterpret_cast<int32_t*>(take(4 * n_chunk));
  t.chunk_off = reinterpret_cast<int32_t*>(take(4 * n_chunk));
  t.row = row;
  t.n_pops = q.lay.n_pops;
  if (a) *a = t;
  return at;
}

// byte size of the scratch and, when base != null, its carving
size_t carve(const sai_vcf_query& q, int64_t len, char* base, Scratch* s, int n_chrom = -1) {
  const size_t n_seg = (size_t)((len + kSegBytes - 1) / kSegBytes) + 1;
  const size_t n_line = (size_t)len + 1;
  const size_t n_chunk = n_line / kLinesPerChunk + 2;
  size_t at = 0;
  auto take = [&](size_t bytes) {
    char* p = base ? base + at : nullptr;
    at += al(bytes);
    return p;
  };
  Scratch t;
  t.info = reinterpret_cast<SliceInfo*>(take(sizeof(SliceInfo)));
  t.seg_cnt = reinterpret_cast<int32_t*>(take(4 * n_seg));
  t.seg_off = reinterpret_cast<int32_t*>(take(4 * n_seg));
  t.line_end = reinterpret_cast<int32_t*>(take(4 * n_line));
  t.rec_samp = reinterpret_cast<int32_t*>(take(4 * n_line));
  t.rec_end = reinterpret_cast<int32_t*>(take(4 * n_line));
  t.rec_pos = reinterpret_cast<int32_t*>(take(4 * n_line));
  t.rec_meta = reinterpret_cast<int32_t*>(take(4 * n_line));
  t.chunk_cnt = reinterpret_cast<int32_t*>(take(4 * n_chunk));
  t.chunk_off = reinterpret_cast<int32_t*>(take(4 * n_chunk));
  t.kept = t.line_end;
  t.fields = reinterpret_cast<int32_t*>(take(4 * (size_t)geno_warps() * (size_t)(q.max_column + 1)));
  t.rec_chrom = nullptr, t.rec_span = nullptr, t.bnd = t.seg_k = nullptr, t.seg_site = t.seg_gap = nullptr;
  if (n_chrom >= 0) {
    t.rec_chrom = reinterpret_cast<int32_t*>(take(4 * n_line));
    t.rec_span = reinterpret_cast<uint32_t*>(take(4 * n_line));
    t.bnd = reinterpret_cast<int32_t*>(take(4 * ((size_t)n_chrom + 1)));
    t.seg_k = reinterpret_cast<int32_t*>(take(4 * ((size_t)n_chrom + 2)));
    t.seg_site = reinterpret_cast<int64_t*>(take(8 * ((size_t)n_chrom + 2)));
    t.seg_gap = reinterpret_cast<int64_t*>(take(8 * ((size_t)n_chrom + 2)));
  }
  if (s) *s = t;
  return at;
}

// ---- block-wide exclusive scan of one int per thread (blockDim.x multiple of 32, <= 1024) ----
__device__ int block_excl_scan(int v, int* total) {
  __shared__ int warp_sum[32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int x = v;
  for (int d = 1; d < 32; d <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, d);
    if (lane >= d) x += y;
  }
  if (lane == 31) warp_sum[w] = x;
  __syncthreads();
  if (w == 0) {
    int s = lane < nw ? warp_sum[lane] : 0;
    for (int d = 1; d < 32; d <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, s, d);
      if (lane >= d) s += y;
    }
    if (lane < nw) warp_sum[lane] = s;  // inclusive
  }
  __syncthreads();
  const int before = (w > 0 ? warp_sum[w - 1] : 0) + x - v;
  *total = warp_sum[nw - 1];
  __syncthreads();  // warp_sum is reused by the next call
  return before;
}

// ---- 1. newline index ----------------------------------------------------------------------
// 32 bytes per thread: bitmask of '\n' (the slot base is 256-byte aligned and segments are 8 KB,
// so the two 16-byte loads are aligned)
__device__ inline uint32_t nl_mask32(const char* text, int64_t len, int64_t at) {
  uint32_t m = 0;
  if (at + 32 <= len) {
    const uint4* p = reinterpret_cast<const uint4*>(text + at);
    const uint4 a = __ldg(p), b = __ldg(p + 1);
    const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int k = 0; k < 8; ++k)
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (((w[k] >> (8 * c)) & 0xff) == '\n') m |= 1u << (4 * k + c);
  } else {
    for (int k = 0; k < 32 && at + k < len; ++k)
      if (text[at + k] == '\n') m |= 1u << k;
  }
  return m;
}

__global__ void __launch_bounds__(256) k_nl_count(const char* __restrict__ text, int64_t len, Scratch s) {
  const int64_t at = (int64_t)blockIdx.x * kSegBytes + 32 * threadIdx.x;
  const int c = at < len ? __popc(nl_mask32(text, len, at)) : 0;
  int total;
  block_excl_scan(c, &total);
  if (threadIdx.x == 0) s.seg_cnt[blockIdx.x] = total;
}

// exclusive scan of n ints by one block; *total (optional) = sum
__device__ void scan_one_block(const int32_t* in, int32_t* out, int n, int32_t* total) {
  int carry = 0;
  for (int base = 0; base < n; base += blockDim.x) {
    const int i = base + threadIdx.x;
    const int v = i < n ? in[i] : 0;
    int sum;
    const int ex = block_excl_scan(v, &sum);
    if (i < n) out[i] = carry + ex;
    carry += sum;
  }
  if (total && threadIdx.x == 0) *total = carry;
}

__global__ void __launch_bounds__(1024) k_seg_scan(int n_seg, Scratch s) {
  scan_one_block(s.seg_cnt, s.seg_off, n_seg, &s.info->n_lines);
}

__global__ void __launch_bounds__(256) k_nl_write(const char* __restrict__ text, int64_t len, Scratch s) {
  const int64_t at = (int64_t)blockIdx.x * kSegBytes + 32 * threadIdx.x;
  uint32_t m = at < len ? nl_mask32(text, len, at) : 0;
  int total;
  int r = s.seg_off[blockIdx.x] + block_excl_scan(__popc(m), &total);
  while (m) {
    const int b = __ffs(m) - 1;
    m &= m - 1;
    s.line_end[r++] = (int32_t)(at + b);
  }
}

// ---- 2. record pass ---------------------------------------------------------------------------
// the first nine tabs of the line [ls, le) into T (warp-cooperative); returns how many there are
__device__ inline int find_tabs(const char* __restrict__ text, int32_t ls, int32_t le, int32_t* T, int lane) {
  int n_tab = 0;
  for (int32_t c = ls; c < le && n_tab < 9; c += 32) {
    const bool t = c + lane < le && text[c + lane] == '\t';
    const uint32_t m = __ballot_sync(0xffffffffu, t);
    const int r = n_tab + __popc(m & ((1u << lane) - 1));
    if (t && r < 9) T[r] = c + lane;
    n_tab += __popc(m);
  }
  __syncwarp();
  return n_tab;
}

__device__ inline int64_t parse_pos(const char* __restrict__ text, const int32_t* T) {
  int64_t pos = 0;
  for (int32_t p = T[0] + 1; p < T[1]; ++p)
    pos = (int64_t)((uint64_t)pos * 10u + (uint64_t)(int64_t)((signed char)text[p] - '0'));
  return pos;
}

// rec_meta of a record whose CHROM (and region) matched: the ancestral-allele entries
// [anc_lo, anc_hi) of anc_pos / anc_allele decide keep and flip (no table: anc_lo == anc_hi == -1),
// then the index of the first FORMAT key that is exactly "GT" (0 if none)
__device__ inline int record_meta(const char* __restrict__ text, const int32_t* T, int64_t pos, const int32_t* anc_pos,
                                  const char* anc_allele, int64_t anc_lo, int64_t anc_hi) {
  bool keep = true, flip = false;
  if (anc_lo >= 0) {
    const int32_t key = (int32_t)pos;
    int64_t lo = anc_lo, hi = anc_hi;  // lower_bound
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (anc_pos[mid] < key) lo = mid + 1; else hi = mid;
    }
    if (lo == anc_hi || anc_pos[lo] != key) {
      keep = false;
    } else {
      const char* a = anc_allele + 8 * lo;
      int alen = 0;
      while (alen < 8 && a[alen]) ++alen;
      const int32_t ref = T[2] + 1, ref_len = T[3] - ref;
      const int32_t alt = T[3] + 1;
      int32_t alt_end = T[4];
      for (int32_t p = alt; p < T[4]; ++p)
        if (text[p] == ',') {
          alt_end = p;
          break;
        }
      bool is_ref = ref_len == alen, is_alt = alt_end - alt == alen;
      for (int k = 0; k < alen; ++k) {
        is_ref = is_ref && text[ref + k] == a[k];
        is_alt = is_alt && text[alt + k] == a[k];
      }
      if (!is_ref && !is_alt) keep = false;
      flip = is_alt;
    }
  }
  if (!keep) return 0;
  int gi = 0, k = 0;
  for (int32_t p = T[7] + 1; p < T[8];) {
    int32_t ke = p;
    while (ke < T[8] && text[ke] != ':') ++ke;
    if (ke - p == 2 && text[p] == 'G' && text[p + 1] == 'T') {
      gi = k;
      break;
    }
    p = ke + 1;
    ++k;
  }
  return 1 | (flip ? 2 : 0) | (gi << 2);
}

__device__ inline void line_bounds(const char* __restrict__ text, const Scratch& s, int64_t i, int32_t* ls, int32_t* le) {
  *ls = i > 0 ? s.line_end[i - 1] + 1 : 0;
  *le = s.line_end[i];
  if (*le > *ls && text[*le - 1] == '\r') --*le;
}

__global__ void __launch_bounds__(256) k_records(const char* __restrict__ text, const __grid_constant__ sai_vcf_query q,
                                                 Scratch s) {
  __shared__ int32_t tabs[kWarpsPerBlock][9];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int n_lines = s.info->n_lines;
  const int64_t n_warps = (int64_t)gridDim.x * kWarpsPerBlock;
  for (int64_t i = (int64_t)blockIdx.x * kWarpsPerBlock + wib; i < n_lines; i += n_warps) {
    int32_t ls, le;
    line_bounds(text, s, i, &ls, &le);
    int meta = 0, samp = 0, pos32 = 0;
    if (le > ls && text[ls] != '#') {
      const int n_tab = find_tabs(text, ls, le, tabs[wib], lane);
      if (lane == 0 && n_tab >= 9) {
        const int32_t* T = tabs[wib];
        bool keep = T[0] - ls == q.chrom_len;
        for (int k = 0; keep && k < q.chrom_len; ++k) keep = text[ls + k] == q.chrom[k];
        const int64_t pos = parse_pos(text, T);
        if (keep && q.start <= q.end && (pos < q.start || pos > q.end)) keep = false;
        if (keep)
          meta = record_meta(text, T, pos, q.anc_pos, q.anc_allele, q.n_anc > 0 ? 0 : -1, q.n_anc > 0 ? q.n_anc : -1);
        samp = T[8] + 1;
        pos32 = (int32_t)pos;
      }
    }
    if (lane == 0) {
      s.rec_meta[i] = meta;
      s.rec_samp[i] = samp;
      s.rec_end[i] = le;
      s.rec_pos[i] = pos32;
    }
    __syncwarp();
  }
}

// Genome record pass: CHROM looked up in the chromosome table (hashed into shared memory), every
// record of a listed chromosome noted for its span (rec_chrom, rec_span: POS read as
// sai_vcf_chrom_span reads it, any number of fields), the ancestral-allele search confined to the
// chromosome's own entries.
__global__ void __launch_bounds__(256) k_records_genome(const char* __restrict__ text,
                                                        const __grid_constant__ VcfGenomeQuery g, Scratch s) {
  __shared__ int32_t tabs[kWarpsPerBlock][9];
  __shared__ uint2 table[kChromHashSlots];
  for (int i = threadIdx.x; i < kChromHashSlots; i += blockDim.x)
    table[i] = make_uint2(g.hash[2 * i], g.hash[2 * i + 1]);
  __syncthreads();
  const sai_vcf_query& q = g.q;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int n_lines = s.info->n_lines;
  const int64_t n_warps = (int64_t)gridDim.x * kWarpsPerBlock;
  for (int64_t i = (int64_t)blockIdx.x * kWarpsPerBlock + wib; i < n_lines; i += n_warps) {
    int32_t ls, le;
    line_bounds(text, s, i, &ls, &le);
    int meta = 0, samp = 0, pos32 = 0, chrom = -1;
    uint32_t span = 0;
    if (le > ls && text[ls] != '#') {
      const int n_tab = find_tabs(text, ls, le, tabs[wib], lane);
      if (lane == 0 && n_tab >= 1) {
        const int32_t* T = tabs[wib];
        const int n = T[0] - ls;
        const uint32_t h = chrom_hash(text + ls, n);
        for (uint32_t slot = h & (kChromHashSlots - 1);; slot = (slot + 1) & (kChromHashSlots - 1)) {
          const uint2 e = table[slot];
          if (e.y == 0) break;
          if (e.x != h) continue;
          const int c = (int)e.y - 1;
          const int32_t a = g.name_off[c];
          bool same = g.name_off[c + 1] - a == n;
          for (int k = 0; same && k < n; ++k) same = text[ls + k] == g.names[a + k];
          if (same) {
            chrom = c;
            break;
          }
        }
        if (chrom >= 0) {
          uint64_t sp = 0;  // sai_vcf_chrom_span: the digits behind the first tab
          for (int32_t p = T[0] + 1; p < le && text[p] >= '0' && text[p] <= '9'; ++p) sp = sp * 10 + (text[p] - '0');
          span = (uint32_t)sp;
          if (n_tab >= 9) {
            const int64_t pos = parse_pos(text, T);
            meta = q.n_anc > 0 ? record_meta(text, T, pos, q.anc_pos, q.anc_allele, g.anc_off[chrom], g.anc_off[chrom + 1])
                               : record_meta(text, T, pos, nullptr, nullptr, -1, -1);
            samp = T[8] + 1;
            pos32 = (int32_t)pos;
          }
        }
      }
    }
    if (lane == 0) {
      s.rec_meta[i] = meta;
      s.rec_samp[i] = samp;
      s.rec_end[i] = le;
      s.rec_pos[i] = pos32;
      s.rec_chrom[i] = chrom;
      s.rec_span[i] = span;
    }
    __syncwarp();
  }
}

// ---- 3. site numbering ------------------------------------------------------------------------
// Genome parse: also the spans.  The lines of a warp are consecutive, so among the lanes of one
// chromosome the lowest holds its first record and the highest its last: one atomic each per warp.
template <bool kGenome = false>
__global__ void __launch_bounds__(kLinesPerChunk) k_keep_count(Scratch s, const VcfGenomeState* gs, VcfChromDev* chroms) {
  const int n_lines = s.info->n_lines;
  const int n_chunk = (n_lines + kLinesPerChunk - 1) / kLinesPerChunk;
  for (int c = blockIdx.x; c < n_chunk; c += gridDim.x) {
    const int i = c * kLinesPerChunk + threadIdx.x;
    int total;
    block_excl_scan(i < n_lines ? (s.rec_meta[i] & 1) : 0, &total);
    if (threadIdx.x == 0) s.chunk_cnt[c] = total;
    if constexpr (kGenome) {
      const int ch = i < n_lines ? s.rec_chrom[i] : -1;
      const uint32_t same = __match_any_sync(0xffffffffu, ch);
      const int lane = threadIdx.x & 31;
      if (ch >= 0) {
        const unsigned long long key = ((unsigned long long)(gs->lines + i) << 32) | s.rec_span[i];
        if (lane == __ffs(same) - 1) {
          atomicAdd(reinterpret_cast<unsigned long long*>(&chroms[ch].n_records), (unsigned long long)__popc(same));
          atomicMin(&chroms[ch].first_key, key);
        }
        if (lane == 31 - __clz(same)) atomicMax(&chroms[ch].last_key, key);
      }
    }
  }
}

template <bool kGenome = false>
__global__ void __launch_bounds__(1024) k_keep_scan(Scratch s, sai_vcf_state* st, int64_t site_cap) {
  const int n_chunk = (s.info->n_lines + kLinesPerChunk - 1) / kLinesPerChunk;
  scan_one_block(s.chunk_cnt, s.chunk_off, n_chunk, &s.info->n_kept);
  __syncthreads();
  if (threadIdx.x == 0) {
    const int64_t base = st->n_sites;
    s.info->site_base = base;
    if constexpr (kGenome) {
      s.info->n_bnd = 0;  // k_genome_plan numbers the sites
    } else {
      st->n_sites = base + s.info->n_kept;
      if (base + s.info->n_kept > site_cap) st->overflow = 1;
    }
  }
}

template <bool kGenome = false>
__global__ void __launch_bounds__(kLinesPerChunk) k_keep_write(Scratch s, int32_t* __restrict__ pos, int64_t site_cap) {
  const int n_lines = s.info->n_lines;
  const int n_chunk = (n_lines + kLinesPerChunk - 1) / kLinesPerChunk;
  const int64_t base = s.info->site_base;
  for (int c = blockIdx.x; c < n_chunk; c += gridDim.x) {
    const int i = c * kLinesPerChunk + threadIdx.x;
    const int keep = i < n_lines ? (s.rec_meta[i] & 1) : 0;
    int total;
    const int k = s.chunk_off[c] + block_excl_scan(keep, &total);
    if (keep) {
      s.kept[k] = i;
      if (!kGenome && base + k < site_cap) pos[base + k] = s.rec_pos[i];  // genome: k_genotypes writes pos
    }
  }
}

// genome: the kept records that start a run of one chromosome (the first of the slice continues the
// last chromosome of the previous slices or starts one).  More starts than chromosomes: some
// chromosome resumes, which k_genome_plan reports.
__global__ void __launch_bounds__(256) k_genome_bounds(Scratch s, const VcfGenomeState* gs, int32_t n_chrom) {
  const int n_kept = s.info->n_kept;
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n_kept; k += gridDim.x * blockDim.x) {
    const int c = s.rec_chrom[s.kept[k]];
    const int prev = k > 0 ? s.rec_chrom[s.kept[k - 1]] : gs->last_chrom;
    if (c != prev) {
      const int r = atomicAdd(&s.info->n_bnd, 1);
      if (r <= n_chrom) s.bnd[r] = k;
    }
  }
}

// genome: one thread lays the slice's runs out -- a run that starts a chromosome begins on the next
// tile boundary -- and keeps the per-chromosome site ranges and the running state.  Runs are as rare
// as chromosome changes, so this is a short sequential pass.
__global__ void k_genome_plan(Scratch s, sai_vcf_state* st, VcfGenomeState* gs, VcfChromDev* chroms, int32_t n_chrom,
                              int64_t site_cap) {
  if (threadIdx.x != 0) return;
  SliceInfo& I = *s.info;
  gs->lines += I.n_lines;
  I.n_seg = 0;
  if (gs->noncontiguous || I.n_kept == 0) return;
  const int nb = I.n_bnd;
  if (nb > n_chrom) {
    gs->noncontiguous = 1;
    return;
  }
  for (int a = 1; a < nb; ++a) {  // insertion sort: the starts were appended in any order
    const int v = s.bnd[a];
    int b = a - 1;
    for (; b >= 0 && s.bnd[b] > v; --b) s.bnd[b + 1] = s.bnd[b];
    s.bnd[b + 1] = v;
  }
  int64_t end = st->n_sites;  // one past the last site so far
  int cur = gs->last_chrom;
  int n_seg = 0, at = 0;
  if (nb == 0 || s.bnd[0] > 0) {  // the slice continues the last run
    s.seg_k[0] = 0;
    s.seg_site[0] = s.seg_gap[0] = end;
    n_seg = 1;
  }
  for (int j = 0; j <= nb; ++j) {
    const int k = j < nb ? s.bnd[j] : I.n_kept;
    if (k > at && cur >= 0) {  // close the run [at, k) of `cur`
      chroms[cur].n_sites += k - at;
      end += k - at;
    }
    if (j == nb) break;
    cur = s.rec_chrom[s.kept[k]];
    if (chroms[cur].first_site >= 0) {
      gs->noncontiguous = 1;
      return;
    }
    s.seg_gap[n_seg] = end;
    end = (end + kTile - 1) / kTile * kTile;
    chroms[cur].first_site = end;
    s.seg_k[n_seg] = k;
    s.seg_site[n_seg] = end;
    ++n_seg;
    at = k;
  }
  I.n_seg = n_seg;
  st->n_sites = end;
  gs->last_chrom = cur;
  if (end > site_cap) st->overflow = 1;
}

// ---- 4. genotype pass -------------------------------------------------------------------------
// gt_sum of vcf_parse.cu: GT sub-field of the field at p (ends at a tab or at lend), cut / padded
// to `ploidy` alleles, "." and junk = -1, flipped |a - 1|, summed, clamped to int8
__device__ inline int gt_sum_dev(const char* p, const char* lend, int gt_index, int ploidy, bool flip) {
  for (int k = 0; k < gt_index; ++k) {
    while (p < lend && *p != ':' && *p != '\t') ++p;
    if (p < lend && *p == ':') ++p;
  }
  int sum = 0;
  bool open = p < lend && *p != '\t' && *p != ':';
  for (int n = 0; n < ploidy; ++n) {
    int a = -1;
    if (open) {
      int v = 0;
      bool digits = false, junk = false;
      while (p < lend) {
        const char c = *p;
        if (c == '/' || c == '|' || c == ':' || c == '\t') break;
        if (c >= '0' && c <= '9' && !junk) {
          v = v * 10 + (c - '0');
          digits = true;
        } else {
          junk = true;
        }
        ++p;
      }
      if (digits && !junk) a = v;
      if (p < lend && (*p == '/' || *p == '|'))
        ++p;
      else
        open = false;
    }
    if (flip) a = a > 0 ? a - 1 : 1 - a;
    sum += a;
  }
  return sum < -128 ? -128 : (sum > 127 ? 127 : sum);
}

__device__ inline uint32_t* word_at(void* tiles, int pps, int64_t site, int w) {
  const int64_t T = site >> 5;
  const int sl = (int)(site & 31);
  return reinterpret_cast<uint32_t*>(static_cast<char*>(tiles) + ((T * pps + (w >> 1)) * 32 + sl) * 8 + (w & 1) * 4);
}

// genome parse: the site of the slice's kept record k (its run's site plus its place in the run)
__device__ inline int64_t genome_site(const Scratch& s, int n_seg, int64_t k) {
  int lo = 0, hi = n_seg - 1;  // the last run that starts at or before k
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (s.seg_k[mid] <= k) lo = mid; else hi = mid - 1;
  }
  return s.seg_site[lo] + (k - s.seg_k[lo]);
}

// kNeg: also the negative-value table.  Per (record, population) the lanes' missing calls are
// ranked with one ballot per group (individual order), staged in the warp's `pending` row, and
// copied to the session buffer at an offset reserved with one atomic; the count goes to `cnt`.
template <bool kGenome = false, bool kNeg = false>
__global__ void __launch_bounds__(256) k_genotypes(const char* __restrict__ text, const __grid_constant__ sai_vcf_query q,
                                                   Scratch s, void* __restrict__ tiles, int32_t* __restrict__ pos,
                                                   int64_t site_cap, sai_vcf_state* st, const NegArgs na) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  const int64_t n_warps = (int64_t)gridDim.x * kWarpsPerBlock;
  const int n_kept = kGenome && s.info->n_seg == 0 ? 0 : s.info->n_kept;  // genome: no runs = nothing to write
  const int64_t base = s.info->site_base;
  const int n_seg = kGenome ? s.info->n_seg : 0;
  const int row = q.max_column + 1;
  int32_t* fo = s.fields + warp * row;
  int2* const pend = na.pending + warp * na.row;  // kNeg
  const int pps = q.lay.pairs_per_site;
  for (int64_t k = warp; k < n_kept; k += n_warps) {
    const int64_t site = kGenome ? genome_site(s, n_seg, k) : base + k;
    if (site >= site_cap) break;  // reported through st->overflow (sites grow with k)
    const int line = s.kept[k];
    if (kGenome && lane == 0) pos[site] = s.rec_pos[line];
    const int meta = s.rec_meta[line];
    const bool flip = (meta & 2) != 0;
    const int gi = meta >> 2;
    const char* S = text + s.rec_samp[line];
    const int32_t L = s.rec_end[line] - s.rec_samp[line];  // bytes of the sample columns (>= 0)
    const char* lend = S + L;
    // regular record: tabs exactly at offsets 3, 7, 11, ... -> field c at 4c
    bool regular = gi == 0 && L > 0 && ((L + 1) & 3) == 0;
    for (int32_t c = 0; regular && c < L; c += 32) {
      const int32_t i = c + lane;
      const bool bad = i < L && ((S[i] == '\t') != ((i & 3) == 3));
      if (__any_sync(0xffffffffu, bad)) regular = false;
    }
    int32_t n_fields;
    if (regular) {
      n_fields = (L + 1) >> 2;
    } else {
      // field offsets of columns 0..max_column; a field exists behind every tab (possibly empty)
      n_fields = L > 0 ? 1 : 0;
      if (lane == 0 && L > 0) fo[0] = 0;
      for (int32_t c = 0; c < L && n_fields < row; c += 32) {
        const int32_t i = c + lane;
        const bool t = i < L && S[i] == '\t';
        const uint32_t m = __ballot_sync(0xffffffffu, t);
        const int r = n_fields + __popc(m & ((1u << lane) - 1));
        if (t && r < row) fo[r] = i + 1;
        n_fields += __popc(m);
      }
      __syncwarp();
    }
    int col_base = 0;
    for (int p = 0; p < q.lay.n_pops; ++p) {
      const sai_pop_layout& P = q.lay.pop[p];
      const int B = P.bits, miss = (1 << B) - 1;
      int vmax = 0;
      int n_neg = 0;  // kNeg: missing calls of the record in this population so far
      for (int g = 0; g < P.n_groups; ++g) {
        const int ind = 32 * g + lane;
        uint32_t code = (uint32_t)miss;
        int neg = 0;
        if (ind < P.n_samples) {
          const int col = q.sample_column[col_base + ind];
          int v;
          if (col >= n_fields) {
            v = -P.ploidy;  // column absent: all alleles missing, never flipped
          } else {
            const int32_t f = regular ? 4 * col : fo[col];
            v = gt_sum_dev(S + f, lend, gi, P.ploidy, flip);
          }
          if (v >= 0) {
            code = (uint32_t)v;
            vmax = max(vmax, v);
          }
          if constexpr (kNeg) neg = min(v, 0);
        }
        const int w0 = 2 * P.pair_off + g * B;
        for (int b = 0; b < B; ++b) {
          const uint32_t word = __ballot_sync(0xffffffffu, (code >> b) & 1u);
          if (lane == b) *word_at(tiles, pps, site, w0 + b) = word;
        }
        if constexpr (kNeg) {
          const uint32_t m = __ballot_sync(0xffffffffu, neg < 0);
          if (neg < 0) pend[n_neg + __popc(m & ((1u << lane) - 1))] = make_int2(ind, neg);
          n_neg += __popc(m);
        }
      }
      if constexpr (kNeg) {
        const int64_t item = (int64_t)p * n_kept + k;
        uint32_t rel = 0;
        if (lane == 0) {
          if (n_neg > 0)
            rel = (uint32_t)(atomicAdd(&na.t.state->n, (unsigned long long)n_neg) - na.t.state->slice_base);
          na.cnt[item] = n_neg;
          na.at[item] = rel;
        }
        rel = __shfl_sync(0xffffffffu, rel, 0);
        __syncwarp();  // the pending row is complete
        const int64_t d0 = (int64_t)(na.t.state->slice_base + rel);
        for (int e = lane; e < n_neg; e += 32) {
          const int64_t d = d0 + e;
          if (d < na.t.cap) {
            const int2 x = pend[e];
            na.t.ind[d] = x.x;
            na.t.val[d] = x.y;
          }
        }
        __syncwarp();  // the row is reused by the next population
      }
      if ((P.n_groups * B) & 1)
        if (lane == 0) *word_at(tiles, pps, site, 2 * P.pair_off + P.n_groups * B) = 0u;  // the pad word
      for (int d = 16; d > 0; d >>= 1) vmax = max(vmax, __shfl_xor_sync(0xffffffffu, vmax, d));
      if (lane == 0 && vmax > P.ploidy) atomicMax(&st->vmax[p], vmax);
      col_base += P.n_samples;
    }
  }
}

// ---- 5. padding sites behind the last site, to the end of its tile -----------------------------
__device__ inline void pad_sites(const sai_layout& lay, void* tiles, int64_t lo, int64_t hi) {
  const int n_words = 2 * lay.pairs_per_site;
  for (int64_t x = threadIdx.x; x < (hi - lo) * n_words; x += blockDim.x) {
    const int64_t site = lo + x / n_words;
    const int w = (int)(x % n_words);
    int p = 0;
    while (p + 1 < lay.n_pops && w >= 2 * lay.pop[p + 1].pair_off) ++p;
    const sai_pop_layout& P = lay.pop[p];
    *word_at(tiles, lay.pairs_per_site, site, w) = (w - 2 * P.pair_off) < P.n_groups * P.bits ? 0xffffffffu : 0u;
  }
}

__global__ void k_pad_tail(const __grid_constant__ sai_layout lay, void* tiles, const sai_vcf_state* st, int64_t site_cap) {
  const int64_t n = st->n_sites;
  if (n > site_cap) return;
  pad_sites(lay, tiles, n, (n + 31) & ~int64_t(31));
}

// genome: also the sites between a chromosome's last site and the tile boundary where the next run of
// the slice starts
__global__ void k_pad_genome(const __grid_constant__ sai_layout lay, void* tiles, const sai_vcf_state* st, Scratch s,
                             int64_t site_cap) {
  const int n_seg = s.info->n_seg;
  for (int j = 0; j < n_seg; ++j)
    if (s.seg_site[j] <= site_cap) pad_sites(lay, tiles, s.seg_gap[j], s.seg_site[j]);
  const int64_t n = st->n_sites;
  if (n <= site_cap) pad_sites(lay, tiles, n, (n + 31) & ~int64_t(31));
}

__global__ void k_genome_init(VcfGenomeState* gs, VcfChromDev* chroms, int32_t n_chrom) {
  for (int c = threadIdx.x; c < n_chrom; c += blockDim.x) chroms[c] = VcfChromDev{~0ull, 0ull, 0, -1, 0};
  if (threadIdx.x == 0) *gs = VcfGenomeState{0, -1, 0};
}

// ---- 6. negative-value table: the slice's entries get their key and their index in it -------------
// The kept records k_genotypes wrote (genome: none without runs) and, for record k, its site and the
// first kept record of its chromosome's run in the slice.
template <bool kGenome>
__device__ inline int neg_kept(const Scratch& s) {
  return kGenome && s.info->n_seg == 0 ? 0 : s.info->n_kept;
}
template <bool kGenome>
__device__ inline int64_t neg_site(const Scratch& s, int64_t k, int* k0) {
  if constexpr (kGenome) {
    const int n_seg = s.info->n_seg;
    int lo = 0, hi = n_seg - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (s.seg_k[mid] <= k) lo = mid; else hi = mid - 1;
    }
    *k0 = s.seg_k[lo];
    return s.seg_site[lo] + (k - s.seg_k[lo]);
  } else {
    *k0 = 0;
    return s.info->site_base + k;
  }
}

__global__ void k_neg_begin(VcfNegDev* d) { d->slice_base = d->n; }

// per 1024 (population, record) items: their count; records past site_cap (not parsed) count 0
template <bool kGenome>
__global__ void __launch_bounds__(1024) k_neg_count(Scratch s, const NegArgs na, int64_t site_cap) {
  const int64_t n_kept = neg_kept<kGenome>(s);
  const int64_t n = n_kept * na.n_pops;
  for (int64_t c = blockIdx.x; c * 1024 < n; c += gridDim.x) {
    const int64_t i = c * 1024 + threadIdx.x;
    int v = 0;
    if (i < n) {
      int k0;
      v = neg_site<kGenome>(s, i % n_kept, &k0) < site_cap ? na.cnt[i] : 0;
      na.cnt[i] = v;
    }
    int total;
    block_excl_scan(v, &total);
    if (threadIdx.x == 0) na.chunk_cnt[c] = total;
  }
}

template <bool kGenome>
__global__ void __launch_bounds__(1024) k_neg_scan(Scratch s, const NegArgs na) {
  const int64_t n = (int64_t)neg_kept<kGenome>(s) * na.n_pops;
  scan_one_block(na.chunk_cnt, na.chunk_off, (int)((n + 1023) / 1024), na.cnt + n);
}

template <bool kGenome>
__global__ void __launch_bounds__(1024) k_neg_excl(Scratch s, const NegArgs na) {
  const int64_t n = (int64_t)neg_kept<kGenome>(s) * na.n_pops;
  for (int64_t c = blockIdx.x; c * 1024 < n; c += gridDim.x) {
    const int64_t i = c * 1024 + threadIdx.x;
    const int v = i < n ? na.cnt[i] : 0;
    int total;
    const int ex = na.chunk_off[c] + block_excl_scan(v, &total);
    if (i < n) na.cnt[i] = ex;
  }
}

// every entry of (population p, record k): chromosome-local site, key, index inside the key =
// entries of the key in earlier slices + entries of the key's earlier records in this slice + rank
template <bool kGenome>
__global__ void __launch_bounds__(256) k_neg_fix(Scratch s, const NegArgs na, const VcfChromDev* chroms) {
  const int64_t n_kept = neg_kept<kGenome>(s);
  const int64_t n = n_kept * na.n_pops;
  const VcfNegSession& t = na.t;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int p = (int)(i / n_kept);
    const int m = min(na.cnt[i + 1] - na.cnt[i], na.row);
    if (m <= 0) continue;
    const int64_t k = i - p * n_kept;
    int k0;
    int64_t site = neg_site<kGenome>(s, k, &k0);
    int c = 0;
    if constexpr (kGenome) {
      c = s.rec_chrom[s.kept[k]];
      site -= chroms[c].first_site;
    }
    const int key = c * na.n_pops + p;
    const int64_t idx = (int64_t)t.count[key] + na.cnt[i] - na.cnt[p * n_kept + k0];
    const int64_t d0 = (int64_t)(t.state->slice_base + na.at[i]);
    for (int e = 0; e < m && d0 + e < t.cap; ++e) {
      t.site[d0 + e] = (int32_t)site;
      t.key[d0 + e] = key;
      t.idx[d0 + e] = (int32_t)(idx + e);
    }
  }
}

// the slice's entries of each (run, population) added to its key's count
template <bool kGenome>
__global__ void k_neg_totals(Scratch s, const NegArgs na) {
  const int64_t n_kept = neg_kept<kGenome>(s);
  if (n_kept == 0) return;
  const int n_run = kGenome ? s.info->n_seg : 1;
  for (int r = threadIdx.x; r < n_run * na.n_pops; r += blockDim.x) {
    const int j = r / na.n_pops, p = r % na.n_pops;
    const int64_t k0 = kGenome ? s.seg_k[j] : 0, k1 = kGenome && j + 1 < n_run ? s.seg_k[j + 1] : n_kept;
    const int c = kGenome ? s.rec_chrom[s.kept[k0]] : 0;
    atomicAdd(&na.t.count[c * na.n_pops + p], (unsigned long long)(na.cnt[p * n_kept + k1] - na.cnt[p * n_kept + k0]));
  }
}

__global__ void k_neg_order(const VcfNegSession t, int64_t n, const int64_t* __restrict__ key_off, int32_t* out_site,
                            int32_t* out_ind, int32_t* out_val) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t d = key_off[t.key[e]] + t.idx[e];
    if (d < 0 || d >= n) continue;
    out_site[d] = t.site[e];
    out_ind[d] = t.ind[e];
    out_val[d] = t.val[e];
  }
}

// the table's kernels of one slice, behind its genotype pass
template <bool kGenome>
int neg_slice(const Scratch& s, const NegArgs& na, const VcfChromDev* chroms, int64_t site_cap, int grid, cudaStream_t st) {
  k_neg_count<kGenome><<<grid, 1024, 0, st>>>(s, na, site_cap);
  k_neg_scan<kGenome><<<1, 1024, 0, st>>>(s, na);
  k_neg_excl<kGenome><<<grid, 1024, 0, st>>>(s, na);
  k_neg_fix<kGenome><<<grid * 4, 256, 0, st>>>(s, na, chroms);
  k_neg_totals<kGenome><<<1, 256, 0, st>>>(s, na);
  SAI_CUDA_CHECK(cudaGetLastError());
  return SAI_OK;
}

}  // namespace

int vcf_chrom_table(const char* names, const int32_t* name_off, int32_t n, uint32_t* table) {
  SAI_REQUIRE(names && name_off && table, "chromosome table: NULL argument");
  SAI_REQUIRE(n >= 1 && n <= SAI_VCF_MAX_CHROMS, "chromosome table: %d names (1..%d)", n, SAI_VCF_MAX_CHROMS);
  memset(table, 0, sizeof(uint32_t) * 2 * kChromHashSlots);
  for (int c = 0; c < n; ++c) {
    const int32_t a = name_off[c], len = name_off[c + 1] - a;
    SAI_REQUIRE(len >= 1 && len <= 255, "chromosome table: name %d of %d bytes (1..255)", c, len);
    const uint32_t h = chrom_hash(names + a, len);
    uint32_t slot = h & (kChromHashSlots - 1);
    for (; table[2 * slot + 1]; slot = (slot + 1) & (kChromHashSlots - 1)) {
      const int o = (int)table[2 * slot + 1] - 1;
      SAI_REQUIRE(!(table[2 * slot] == h && name_off[o + 1] - name_off[o] == len && !memcmp(names + name_off[o], names + a, len)),
                  "chromosome table: %.*s is listed twice", len, names + a);
    }
    table[2 * slot] = h;
    table[2 * slot + 1] = (uint32_t)c + 1;
  }
  return SAI_OK;
}

int vcf_genome_state_init(VcfGenomeState* d_gs, VcfChromDev* d_chroms, int32_t n_chrom, cudaStream_t stream) {
  k_genome_init<<<1, 256, 0, stream>>>(d_gs, d_chroms, n_chrom);
  SAI_CUDA_CHECK(cudaGetLastError());
  return SAI_OK;
}

uint64_t vcf_genome_scratch_bytes(const VcfGenomeQuery& g, int64_t len) {
  return (uint64_t)carve(g.q, len, nullptr, nullptr, g.n_chrom) + 256;
}

uint64_t vcf_neg_scratch_bytes(const sai_vcf_query& q, int64_t len) { return (uint64_t)carve_neg(q, len, nullptr, nullptr); }

int vcf_neg_order(const VcfNegSession& neg, int64_t n, const int64_t* d_key_off, int32_t* out_site, int32_t* out_ind,
                  int32_t* out_val, cudaStream_t st) {
  if (n <= 0) return SAI_OK;
  const int64_t want = (n + 255) / 256, cap = (int64_t)sm_count() * 8;
  k_neg_order<<<(unsigned)(want < cap ? want : cap), 256, 0, st>>>(neg, n, d_key_off, out_site, out_ind, out_val);
  SAI_CUDA_CHECK(cudaGetLastError());
  return SAI_OK;
}

// the scratch of the negative-value table behind the parse scratch (`need` bytes), checked against its size
static int neg_args(const sai_vcf_query& q, int64_t len, void* d_scratch, uint64_t scratch_bytes, size_t need,
                    const VcfNegSession* neg, NegArgs* na) {
  *na = NegArgs{};
  if (!neg) return SAI_OK;
  const size_t extra = carve_neg(q, len, static_cast<char*>(d_scratch) + need, na);
  SAI_REQUIRE(scratch_bytes >= need + extra, "device ingest: scratch of %llu bytes, %zu needed with the negative-value table",
              (unsigned long long)scratch_bytes, need + extra);
  na->t = *neg;
  return SAI_OK;
}

int vcf_tiles_genome(const VcfGenomeQuery& g, const char* d_text, int64_t len, void* d_scratch, uint64_t scratch_bytes,
                     void* d_tiles, int32_t* d_pos, int64_t site_cap, sai_vcf_state* d_state, VcfGenomeState* d_gs,
                     VcfChromDev* d_chroms, const VcfNegSession* neg, cudaStream_t st) {
  SAI_REQUIRE(len >= 0 && len < (int64_t(1) << 31), "vcf_tiles_genome: slice of %lld bytes (at most 2^31 - 1)",
              (long long)len);
  SAI_REQUIRE(site_cap >= 0 && site_cap % kTile == 0, "vcf_tiles_genome: site_cap must be a multiple of 32");
  Scratch s;
  const size_t need = carve(g.q, len, static_cast<char*>(d_scratch), &s, g.n_chrom);
  SAI_REQUIRE(scratch_bytes >= need, "vcf_tiles_genome: scratch of %llu bytes, %zu needed",
              (unsigned long long)scratch_bytes, need);
  NegArgs na;
  if (int rc = neg_args(g.q, len, d_scratch, scratch_bytes, need, neg, &na)) return rc;
  const int n_seg = (int)((len + kSegBytes - 1) / kSegBytes);
  const int grid = sm_count() * 4;
  if (n_seg > 0) {
    k_nl_count<<<n_seg, 256, 0, st>>>(d_text, len, s);
    SAI_CUDA_CHECK(cudaGetLastError());
    k_seg_scan<<<1, 1024, 0, st>>>(n_seg, s);
    k_nl_write<<<n_seg, 256, 0, st>>>(d_text, len, s);
  } else {
    SAI_CUDA_CHECK(cudaMemsetAsync(&s.info->n_lines, 0, sizeof(int32_t), st));
  }
  k_records_genome<<<grid, 32 * kWarpsPerBlock, 0, st>>>(d_text, g, s);
  k_keep_count<true><<<grid, kLinesPerChunk, 0, st>>>(s, d_gs, d_chroms);
  k_keep_scan<true><<<1, 1024, 0, st>>>(s, d_state, site_cap);
  k_keep_write<true><<<grid, kLinesPerChunk, 0, st>>>(s, d_pos, site_cap);
  k_genome_bounds<<<grid, 256, 0, st>>>(s, d_gs, g.n_chrom);
  k_genome_plan<<<1, 32, 0, st>>>(s, d_state, d_gs, d_chroms, g.n_chrom, site_cap);
  if (neg) {
    k_neg_begin<<<1, 1, 0, st>>>(neg->state);
    k_genotypes<true, true><<<grid, 32 * kWarpsPerBlock, 0, st>>>(d_text, g.q, s, d_tiles, d_pos, site_cap, d_state, na);
    if (int rc = neg_slice<true>(s, na, d_chroms, site_cap, grid, st)) return rc;
  } else {
    k_genotypes<true><<<grid, 32 * kWarpsPerBlock, 0, st>>>(d_text, g.q, s, d_tiles, d_pos, site_cap, d_state, na);
  }
  k_pad_genome<<<1, 256, 0, st>>>(g.q.lay, d_tiles, d_state, s, site_cap);
  SAI_CUDA_CHECK(cudaGetLastError());
  return SAI_OK;
}

}  // namespace sai

using namespace sai;

extern "C" {

uint64_t sai_vcf_scratch_bytes(const sai_vcf_query* q, int64_t len) {
  if (!q || len < 0) return 0;
  return (uint64_t)carve(*q, len, nullptr, nullptr) + 256;
}

int sai_vcf_tiles_device(const sai_vcf_query* q, const char* d_text, int64_t len, void* d_scratch,
                         uint64_t scratch_bytes, void* d_tiles, int32_t* d_pos, int64_t site_cap,
                         sai_vcf_state* d_state, void* stream) {
  SAI_REQUIRE(q, "sai_vcf_tiles_device: NULL argument");
  return vcf_tiles_single(*q, d_text, len, d_scratch, scratch_bytes, d_tiles, d_pos, site_cap, d_state, nullptr,
                          static_cast<cudaStream_t>(stream));
}

}  // extern "C"

int sai::vcf_tiles_single(const sai_vcf_query& qr, const char* d_text, int64_t len, void* d_scratch,
                          uint64_t scratch_bytes, void* d_tiles, int32_t* d_pos, int64_t site_cap,
                          sai_vcf_state* d_state, const VcfNegSession* neg, cudaStream_t st) {
  const sai_vcf_query* q = &qr;
  SAI_REQUIRE(d_state && d_scratch && d_tiles && d_pos, "sai_vcf_tiles_device: NULL argument");
  if (int rc = validate_layout(&q->lay)) return rc;
  SAI_REQUIRE(len >= 0 && len < (int64_t(1) << 31), "sai_vcf_tiles_device: slice of %lld bytes (at most 2^31 - 1)",
              (long long)len);
  SAI_REQUIRE(len == 0 || d_text, "sai_vcf_tiles_device: NULL text");
  SAI_REQUIRE(q->chrom_len >= 1 && q->chrom_len < (int)sizeof(q->chrom), "sai_vcf_tiles_device: bad chromosome name");
  SAI_REQUIRE(q->max_column >= 0 && q->sample_column, "sai_vcf_tiles_device: bad sample columns");
  SAI_REQUIRE(q->n_anc == 0 || (q->anc_pos && q->anc_allele), "sai_vcf_tiles_device: bad ancestral-allele table");
  SAI_REQUIRE(site_cap >= 0 && site_cap % kTile == 0, "sai_vcf_tiles_device: site_cap must be a multiple of 32");
  SAI_REQUIRE((reinterpret_cast<uintptr_t>(d_text) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_scratch) & 255) == 0,
              "sai_vcf_tiles_device: text must be 16-byte and scratch 256-byte aligned");
  Scratch s;
  const size_t need = carve(*q, len, static_cast<char*>(d_scratch), &s);
  SAI_REQUIRE(scratch_bytes >= need, "sai_vcf_tiles_device: scratch of %llu bytes, %zu needed",
              (unsigned long long)scratch_bytes, need);
  NegArgs na;
  if (int rc = neg_args(*q, len, d_scratch, scratch_bytes, need, neg, &na)) return rc;
  const int n_seg = (int)((len + kSegBytes - 1) / kSegBytes);
  const int grid = sm_count() * 4;
  if (n_seg > 0) {
    k_nl_count<<<n_seg, 256, 0, st>>>(d_text, len, s);
    SAI_CUDA_CHECK(cudaGetLastError());
    k_seg_scan<<<1, 1024, 0, st>>>(n_seg, s);
    k_nl_write<<<n_seg, 256, 0, st>>>(d_text, len, s);
  } else {
    SAI_CUDA_CHECK(cudaMemsetAsync(&s.info->n_lines, 0, sizeof(int32_t), st));
  }
  k_records<<<grid, 32 * kWarpsPerBlock, 0, st>>>(d_text, *q, s);
  k_keep_count<<<grid, kLinesPerChunk, 0, st>>>(s, nullptr, nullptr);
  k_keep_scan<<<1, 1024, 0, st>>>(s, d_state, site_cap);
  k_keep_write<<<grid, kLinesPerChunk, 0, st>>>(s, d_pos, site_cap);
  if (neg) {
    k_neg_begin<<<1, 1, 0, st>>>(neg->state);
    k_genotypes<false, true><<<grid, 32 * kWarpsPerBlock, 0, st>>>(d_text, *q, s, d_tiles, d_pos, site_cap, d_state, na);
    if (int rc = neg_slice<false>(s, na, nullptr, site_cap, grid, st)) return rc;
  } else {
    k_genotypes<<<grid, 32 * kWarpsPerBlock, 0, st>>>(d_text, *q, s, d_tiles, d_pos, site_cap, d_state, na);
  }
  k_pad_tail<<<1, 256, 0, st>>>(q->lay, d_tiles, d_state, site_cap);
  SAI_CUDA_CHECK(cudaGetLastError());
  return SAI_OK;
}
