// K1: the genotype pass.  One warp owns one 32-site tile, lane == site.
//
// Replaces, per population, the four numpy passes of calc_freq
// (sai/stats/stat_utils.py:45-49) by a carry-save (Harley-Seal) popcount over
// the tile's bit-planes, and -- fused in the epilogue -- the site conditions of
// compute_matching_loci (stat_utils.py:114-166) and UStatistic / QStatistic
// (u_statistic.py:92, q_statistic.py:92).
//
// HBM-bound: every packed byte is read exactly once with coalesced 256-byte
// warp requests (8 bytes per lane); outputs are two 32-bit masks per tile and
// job plus one double per Q-flagged site.
#include <string.h>

#include <algorithm>

#include "common.cuh"
#include "popcount.cuh"
#include "scratch.cuh"
#include "site_cond.cuh"

namespace sai {

// B == 2 population: planes (a = bit0, b = bit1) of one group sit in one pair.
//   num  = popc(a) + 2 popc(b) - 3 popc(a&b),   missing = popc(a&b)
// MODE 0 is the product path (carry-save, 8 loads in flight per lane); MODE 1 (16 loads in
// flight) and MODE 2 (direct POPC per word) exist only in -DSAI_EXPERIMENTS builds (tools/).
template <int MODE>
__device__ __forceinline__ void count_b2(const uint2* __restrict__ col, int n_pairs, int& num,
                                         int& miss) {
  int p = 0;
  int acc_a = 0, acc_b = 0, acc_m = 0;
  if (MODE != 2) {
    SliceCounter ca, cb, cm;
#ifdef SAI_EXPERIMENTS
    if (MODE == 1) {
      for (; p + 16 <= n_pairs; p += 16) {
        uint2 v[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = ld_stream(col + (size_t)(p + i) * kTile);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          uint32_t a[8], b[8], m[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            a[i] = v[8 * h + i].x;
            b[i] = v[8 * h + i].y;
            m[i] = v[8 * h + i].x & v[8 * h + i].y;
          }
          ca.add8(a);
          cb.add8(b);
          cm.add8(m);
        }
      }
    }
#endif
    for (; p + 8 <= n_pairs; p += 8) {
      uint2 v[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = ld_stream(col + (size_t)(p + i) * kTile);
      uint32_t a[8], b[8], m[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        a[i] = v[i].x;
        b[i] = v[i].y;
        m[i] = v[i].x & v[i].y;
      }
      ca.add8(a);
      cb.add8(b);
      cm.add8(m);
    }
    acc_a = ca.total();
    acc_b = cb.total();
    acc_m = cm.total();
  }
  // remainder (and MODE 2): direct popcounts
#pragma unroll 4
  for (; p < n_pairs; ++p) {
    uint2 v = ld_stream(col + (size_t)p * kTile);
    acc_a += __popc(v.x);
    acc_b += __popc(v.y);
    acc_m += __popc(v.x & v.y);
  }
  num = acc_a + 2 * acc_b - 3 * acc_m;
  miss = acc_m;
}

// B == 4 population (values up to 14: high ploidy, or the reference's flipped-missing
// quirk, sai/utils/utils.py:555): a group is two pairs (planes 0,1 | planes 2,3).
//   num = sum_b 2^b popc(plane_b) - 15 popc(and of the planes),   missing = popc(and)
// Same streaming 8-byte loads and carry-save counters as count_b2: 8 loads (4 groups) in
// flight per lane, one counter per plane plus one for the missing mask.
__device__ __forceinline__ void count_b4(const uint2* __restrict__ col, int n_groups, int& num,
                                         int& miss) {
  SliceCounter c0, c1, c2, c3, cm;
  int g = 0;
  for (; g + 4 <= n_groups; g += 4) {
    uint2 v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = ld_stream(col + (size_t)(2 * g + i) * kTile);
    c0.add4(v[0].x, v[2].x, v[4].x, v[6].x);
    c1.add4(v[0].y, v[2].y, v[4].y, v[6].y);
    c2.add4(v[1].x, v[3].x, v[5].x, v[7].x);
    c3.add4(v[1].y, v[3].y, v[5].y, v[7].y);
    cm.add4(v[0].x & v[0].y & v[1].x & v[1].y, v[2].x & v[2].y & v[3].x & v[3].y,
            v[4].x & v[4].y & v[5].x & v[5].y, v[6].x & v[6].y & v[7].x & v[7].y);
  }
  int a0 = c0.total(), a1 = c1.total(), a2 = c2.total(), a3 = c3.total(), am = cm.total();
  for (; g < n_groups; ++g) {
    const uint2 lo = ld_stream(col + (size_t)(2 * g) * kTile);
    const uint2 hi = ld_stream(col + (size_t)(2 * g + 1) * kTile);
    a0 += __popc(lo.x);
    a1 += __popc(lo.y);
    a2 += __popc(hi.x);
    a3 += __popc(hi.y);
    am += __popc(lo.x & lo.y & hi.x & hi.y);
  }
  num = a0 + 2 * a1 + 4 * a2 + 8 * a3 - 15 * am;
  miss = am;
}

// B == 3 population (ploidy 3..6, values up to 6): two groups share three pairs
// (a0,a1 | a2,b0 | b1,b2); an odd last group ends with a zero pad word.
__device__ __forceinline__ void count_b3(const uint2* __restrict__ col, int n_groups, int& num,
                                         int& miss) {
  SliceCounter c0, c1, c2, cm;
  int g = 0;
  for (; g + 4 <= n_groups; g += 4) {
    uint2 v[6];
#pragma unroll
    for (int i = 0; i < 6; ++i) v[i] = ld_stream(col + (size_t)(3 * (g >> 1) + i) * kTile);
    c0.add4(v[0].x, v[1].y, v[3].x, v[4].y);
    c1.add4(v[0].y, v[2].x, v[3].y, v[5].x);
    c2.add4(v[1].x, v[2].y, v[4].x, v[5].y);
    cm.add4(v[0].x & v[0].y & v[1].x, v[1].y & v[2].x & v[2].y, v[3].x & v[3].y & v[4].x,
            v[4].y & v[5].x & v[5].y);
  }
  int a0 = c0.total(), a1 = c1.total(), a2 = c2.total(), am = cm.total();
  const uint32_t* base = reinterpret_cast<const uint32_t*>(col);
  for (; g < n_groups; ++g) {
    uint32_t x[3];
#pragma unroll
    for (int b = 0; b < 3; ++b) {
      const int word = g * 3 + b;  // word w of this lane: pair (w>>1) is 32 lanes * 2 words further on
      x[b] = __ldg(base + (size_t)(word >> 1) * (kTile * 2) + (word & 1));
    }
    a0 += __popc(x[0]);
    a1 += __popc(x[1]);
    a2 += __popc(x[2]);
    am += __popc(x[0] & x[1] & x[2]);
  }
  num = a0 + 2 * a1 + 4 * a2 - 7 * am;
  miss = am;
}

// B = 5..8 (per-individual values above 14: multi-allelic genotype indices >= 8): plain per-word
// path, the planes of a group back to back.  Correct for any B; not tuned -- such data is rare.
__device__ __forceinline__ void count_wide(const uint2* __restrict__ col, int n_groups, int B, int& num, int& miss) {
  const uint32_t* base = reinterpret_cast<const uint32_t*>(col);
  const int all = (1 << B) - 1;
  int acc = 0, accm = 0;
  for (int g = 0; g < n_groups; ++g) {
    uint32_t andw = 0xffffffffu;
    int s = 0;
    for (int b = 0; b < B; ++b) {
      const int word = g * B + b;  // word w of this lane: pair (w >> 1) is 32 lanes * 2 words further on
      const uint32_t x = __ldg(base + (size_t)(word >> 1) * (kTile * 2) + (word & 1));
      s += __popc(x) << b;
      andw &= x;
    }
    const int m = __popc(andw);
    acc += s - all * m;
    accm += m;
  }
  num = acc;
  miss = accm;
}

// (num, called) of one population at the lane's site; col = the population's first pair of the tile
template <int MODE>
__device__ __forceinline__ void count_pop(const sai_pop_layout& L, const uint2* __restrict__ col, int& num,
                                          int& called) {
  int miss;
  if (L.bits == 2)
    count_b2<MODE>(col, L.n_pairs, num, miss);
  else if (L.bits == 4)
    count_b4(col, L.n_groups, num, miss);
  else if (L.bits == 3)
    count_b3(col, L.n_groups, num, miss);
  else
    count_wide(col, L.n_groups, L.bits, num, miss);
  called = L.n_groups * 32 - miss;
}

// ---- host side of the integer fast path (site_cond.cuh) ----------------------------
namespace {
// first n in [0, d + 1] for which pred(n) holds; pred must be monotone (false ... false true ... true)
template <typename Pred>
int first_true(int d, Pred pred) {
  int lo = 0, hi = d + 1;
  while (lo < hi) {
    const int mid = lo + (hi - lo) / 2;
    if (pred(mid)) hi = mid; else lo = mid + 1;
  }
  return lo;
}
inline double freq_of(int n, int d) { return (double)n / (double)d; }
// {n in [0, d] : op(freq(n), y)} as [lo, hi] (empty: lo > hi); freq is non-decreasing in n
void op_interval(int op, double y, int d, int32_t& lo, int32_t& hi) {
  const int ge = first_true(d, [&](int n) { return freq_of(n, d) >= y; });  // first n with freq >= y
  const int gt = first_true(d, [&](int n) { return freq_of(n, d) > y; });   // first n with freq >  y
  switch (op) {
    case SAI_OP_EQ: lo = ge, hi = gt - 1; break;
    case SAI_OP_LT: lo = 0, hi = ge - 1; break;
    case SAI_OP_GT: lo = gt, hi = d; break;
    case SAI_OP_LE: lo = 0, hi = gt - 1; break;
    default: lo = ge, hi = d; break;
  }
  if (y != y) lo = 1, hi = 0;  // NaN compares false (cannot pass validation, but stay exact)
}
}  // namespace

void build_job_fast(const sai_layout& lay, const sai_job& J, JobFast& F) {
  memset(&F, 0, sizeof(F));
  auto den = [&](int pop) { return (int64_t)lay.pop[pop].n_samples * lay.pop[pop].ploidy; };
  int64_t dmax = std::max(den(J.ref_pop), den(J.tgt_pop));
  for (int k = 0; k < J.n_src; ++k) dmax = std::max(dmax, den(J.src_pop[k]));
  if (dmax >= (1ll << 30)) return;  // F.ok = 0: always the division path
  const int dr = (int)den(J.ref_pop), dt = (int)den(J.tgt_pop);
  F.den_ref = dr;
  F.den_tgt = dt;
  // tgt_freq > x  <=> n >= tgt_min;   1 - tgt_freq > x  <=> n <= tgt_inv_max (non-increasing in n)
  F.tgt_min = first_true(dt, [&](int n) { return freq_of(n, dt) > J.x; });
  F.tgt_inv_max = first_true(dt, [&](int n) { return !(1.0 - freq_of(n, dt) > J.x); }) - 1;
  const sai_cond* cs[2] = {&J.u, &J.q};
  CondFast* fs[2] = {&F.u, &F.q};
  for (int c = 0; c < 2; ++c) {
    const sai_cond& C = *cs[c];
    CondFast& X = *fs[c];
    // ref_freq < w  <=> n <= ref_max;   1 - ref_freq < w  <=> n >= ref_inv_min
    X.ref_max = first_true(dr, [&](int n) { return !(freq_of(n, dr) < C.w); }) - 1;
    X.ref_inv_min = first_true(dr, [&](int n) { return 1.0 - freq_of(n, dr) < C.w; });
    for (int k = 0; k < J.n_src; ++k) {
      const int ds = (int)den(J.src_pop[k]);
      F.den_src[k] = ds;
      op_interval(C.op[k], C.y[k], ds, X.y_lo[k], X.y_hi[k]);
      op_interval(C.op[k], C.one_minus_y[k], ds, X.f_lo[k], X.f_hi[k]);
    }
  }
  F.ok = 1;
}

// k_site_scan's test of one job: a necessary condition of its source gate (site_gate with
// with_ref == false) on its first source alone.  Where that population is fully called
// (called * ploidy == den) the gate needs its count in one of the n intervals [lo, hi] -- the y and,
// without ancestral alleles, 1 - y intervals of the enabled U / Q conditions; anywhere else the
// site counts as live.
struct ScanTest {
  int32_t pop, den, n;
  int32_t lo[4], hi[4];
};

struct SiteParams {
  sai_layout lay;
  const uint2* packed;  // tile 0
  int64_t tile0, n_tiles, n_tiles_total;
  uint32_t* mask_u;
  uint32_t* mask_q;
  double* qval;
  int64_t qval_stride;
  int32_t* num;
  int32_t* called;
  int64_t count_stride;
  // staged pass only (k_site_scan, k_site_live)
  unsigned long long* counters;  // [0] queue length, [1] batches claimed; zero at launch
  int32_t* queue;                // [n_tiles] live tiles (relative to tile0), in no particular order
  uint32_t gate_pops;            // populations that are a source of a job with U or Q enabled
  int32_t batch_tiles;           // live tiles per batch of k_site_live, 1..kGateTiles
  uint32_t scan_pops;            // populations k_site_scan reads: the first source of each job in scan[]
  int32_t scan_all;              // some job can be live at any site: every tile is queued, nothing read
  int32_t n_scan;
  ScanTest scan[SAI_MAX_JOBS];   // jobs with U or Q enabled and integer intervals
};

constexpr int kSiteWarps = 8;

template <int MODE, bool FUSED>
__global__ void __launch_bounds__(kSiteWarps * 32, MODE == 1 ? 3 : 4)
    k_site(const __grid_constant__ SiteParams P, const __grid_constant__ JobBlock JB,
           const __grid_constant__ JobFastBlock JF) {
  extern __shared__ int s_counts[];  // [warp][2][n_pops][32]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_pops = P.lay.n_pops;
  int* s_num = s_counts + warp * (2 * n_pops * kTile);
  int* s_cal = s_num + n_pops * kTile;
  const int64_t pps = P.lay.pairs_per_site;

  for (int64_t t = (int64_t)blockIdx.x * kSiteWarps + warp; t < P.n_tiles;
       t += (int64_t)gridDim.x * kSiteWarps) {
    const int64_t T = P.tile0 + t;
    const uint2* tile = P.packed + (size_t)T * pps * kTile + lane;
    for (int pi = 0; pi < n_pops; ++pi) {
      const sai_pop_layout& L = P.lay.pop[pi];
      int num, called;
      count_pop<MODE>(L, tile + (size_t)L.pair_off * kTile, num, called);
      s_num[pi * kTile + lane] = num;
      s_cal[pi * kTile + lane] = called;
      if (P.num) {
        const int64_t site = T * kTile + lane;
        P.num[(size_t)pi * P.count_stride + site] = num;
        P.called[(size_t)pi * P.count_stride + site] = called;
      }
    }
    if (FUSED) {
      const int64_t site = T * kTile + lane;
      for (int j = 0; j < JB.n_jobs; ++j) {
        const sai_job& J = JB.job[j];
        SiteFlags f = eval_site_fast(
            JF.job[j], J, P.lay, [&](int pop) { return s_num[pop * kTile + lane]; },
            [&](int pop) { return s_cal[pop * kTile + lane]; });
        const uint32_t mu = __ballot_sync(0xffffffffu, f.u);
        const uint32_t mq = __ballot_sync(0xffffffffu, f.q);
        if (lane == 0) {
          P.mask_u[(size_t)j * P.n_tiles_total + T] = mu;
          P.mask_q[(size_t)j * P.n_tiles_total + T] = mq;
        }
        if (f.q) P.qval[(size_t)j * P.qval_stride + site] = f.q_tgt_freq;
      }
    }
  }
}

// K1 without stored counts: the staged pass.  A site can be flagged only where its sources match
// and its reference frequency is below w (site_gate), and the sources are the smallest operand
// (bench layout: 1 of 80 pairs), so a tile is read in three stages -- the source populations of
// all jobs, the references of the jobs still live, the targets of those still live -- and each
// population at most once.  Stages 2 and 3 read a population only at the sites where a job can
// still hold (gather_sites), unless a tile has more than kGatherSites of them.  Decisions are
// unchanged: the flags of a job come from eval_site_fast, as in k_site, at the sites that passed
// its gates; a job dead on a tile stores zero mask words (and no qval, which exists only at
// Q-flagged sites).
//
// Two kernels.  k_site_scan reads the first source of every job at every tile and tests it against
// interval bounds the host computes in advance (ScanTest, a necessary condition of the source gate):
// a tile where no job can be live gets its zero mask words there, any other is appended to a queue.
// k_site_live runs the three stages on the queued tiles only.  Most tiles are dead (bench data: 77 %) and a live one usually holds a single live site, so
// batching consecutive tiles paid a batch's whole chain of dependent DRAM round trips for about one
// site; batching queued tiles gives each round trip several live tiles' worth of gathers.
//
// Live tiles fall at random and their cost varies, so k_site_live's warps claim batches of
// batch_tiles queue entries from a counter (a static map leaves the busiest warp with ~2x the mean).
// Shared memory holds the counts of every tile of a batch: [warp][tile][2][n_pops][32].
constexpr int kGateTiles = 4;
constexpr int kScanTiles = 8;
constexpr int kGateSmemPerWarp = 6144;  // bounds a batch's shared counts: 4 blocks per SM at any n_pops
// A tile with more live sites than this reads the population whole (n_pairs coalesced loads per
// lane) instead of gathering (per site ceil(n_groups / 32) loads per lane, 32 sectors each).
constexpr int kGatherSites = 8;

// Stage 1: (num, called) of the gate populations at this lane's site of n tiles into the counts of
// each tile.  tile(g) is tile g's first pair at this lane's site and is called by the whole warp.
// 2 planes: pair by pair across the tiles, n loads in flight per lane; other widths tile by tile.
template <int NT, typename TileFn>
__device__ __forceinline__ void count_sources(const SiteParams& P, int n, TileFn tile, int* s_warp, int per_tile,
                                              int lane) {
  const int n_pops = P.lay.n_pops;
  for (uint32_t m = P.gate_pops; m; m &= m - 1) {
    const int pi = __ffs(m) - 1;
    const sai_pop_layout& L = P.lay.pop[pi];
    int* s_num = s_warp + pi * kTile + lane;
    int* s_cal = s_num + n_pops * kTile;
    if (L.bits == 2) {
      int num[NT], miss[NT];
#pragma unroll
      for (int g = 0; g < NT; ++g) num[g] = miss[g] = 0;
      for (int i = 0; i < L.n_pairs; ++i) {
        uint2 v[NT];
#pragma unroll
        for (int g = 0; g < NT; ++g)
          v[g] = g < n ? ld_stream(tile(g) + (size_t)(L.pair_off + i) * kTile) : make_uint2(0u, 0u);
#pragma unroll
        for (int g = 0; g < NT; ++g) {
          const int mm = __popc(v[g].x & v[g].y);
          num[g] += __popc(v[g].x) + 2 * __popc(v[g].y) - 3 * mm;
          miss[g] += mm;
        }
      }
#pragma unroll
      for (int g = 0; g < NT; ++g) {
        if (g < n) {
          s_num[g * per_tile] = num[g];
          s_cal[g * per_tile] = L.n_groups * 32 - miss[g];
        }
      }
    } else {
      for (int g = 0; g < n; ++g)
        count_pop<0>(L, tile(g) + (size_t)L.pair_off * kTile, s_num[g * per_tile], s_cal[g * per_tile]);
    }
  }
}

// Phase A over tiles [tile0, tile0 + n_tiles): one warp takes 32 consecutive tiles per trip, in
// steps of kScanTiles tiles whose loads are in flight together.  Per step and lane, the counts of
// each population in scan_pops at its site of every tile stay in registers, and bit g of site_live
// says whether the ScanTest of some job holds at this lane's site of tile g; a warp-wide OR of it
// gives the tiles of the step that may be live.  Lane g then owns tile g of the trip: it stores the
// tile's zero mask words (32 tiles = one 128-byte store per array and job) or its queue entry, with
// one atomic per trip reserving the trip's entries.  The tests only ever queue a superset of the
// live tiles: k_site_live decides every queued tile exactly, so a tile queued for nothing stores
// zero mask words there.  WIDE: some scanned population has more than two planes (count_pop, whose
// inlined counters need more than 64 registers); otherwise one popcount path for 2-plane groups.
template <bool WIDE>
__global__ void __launch_bounds__(kSiteWarps * 32, WIDE ? 3 : 4)
    k_site_scan(const __grid_constant__ SiteParams P, const __grid_constant__ JobBlock JB) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t pps = P.lay.pairs_per_site;
  for (int64_t t0 = ((int64_t)blockIdx.x * kSiteWarps + warp) * kTile; t0 < P.n_tiles;
       t0 += (int64_t)gridDim.x * kSiteWarps * kTile) {
    const int n = (int)(P.n_tiles - t0 < kTile ? P.n_tiles - t0 : kTile);
    uint32_t live = P.scan_all ? 0xffffffffu : 0u;  // bit g: a job may be live at a site of tile t0 + g
    for (int s0 = 0; s0 < n && !P.scan_all; s0 += kScanTiles) {
      const int ns = n - s0 < kScanTiles ? n - s0 : kScanTiles;
      const uint2* first = P.packed + (size_t)(P.tile0 + t0 + s0) * pps * kTile + lane;
      uint32_t site_live = 0;
      for (uint32_t m = P.scan_pops; m; m &= m - 1) {
        const int pi = __ffs(m) - 1;
        const sai_pop_layout& L = P.lay.pop[pi];
        int num[kScanTiles], called[kScanTiles];
        if (WIDE) {
#pragma unroll
          for (int g = 0; g < kScanTiles; ++g) {
            num[g] = called[g] = 0;
            if (g < ns) count_pop<0>(L, first + ((size_t)g * pps + L.pair_off) * kTile, num[g], called[g]);
          }
        } else {
          int miss[kScanTiles];
#pragma unroll
          for (int g = 0; g < kScanTiles; ++g) num[g] = miss[g] = 0;
          for (int i = 0; i < L.n_pairs; ++i) {
            uint2 v[kScanTiles];
#pragma unroll
            for (int g = 0; g < kScanTiles; ++g)
              v[g] = g < ns ? ld_stream(first + ((size_t)g * pps + L.pair_off + i) * kTile) : make_uint2(0u, 0u);
#pragma unroll
            for (int g = 0; g < kScanTiles; ++g) {
              const int mm = __popc(v[g].x & v[g].y);
              num[g] += __popc(v[g].x) + 2 * __popc(v[g].y) - 3 * mm;
              miss[g] += mm;
            }
          }
#pragma unroll
          for (int g = 0; g < kScanTiles; ++g) called[g] = L.n_groups * 32 - miss[g];
        }
        for (int j = 0; j < P.n_scan; ++j) {
          const ScanTest& T = P.scan[j];
          if (T.pop != pi) continue;
#pragma unroll
          for (int g = 0; g < kScanTiles; ++g) {
            bool ok = called[g] * L.ploidy != T.den;
#pragma unroll
            for (int i = 0; i < 4; ++i) ok = ok || (i < T.n && num[g] >= T.lo[i] && num[g] <= T.hi[i]);
            site_live |= (uint32_t)ok << g;
          }
        }
      }
      live |= (__reduce_or_sync(0xffffffffu, site_live) & ((1u << ns) - 1u)) << s0;
    }
    unsigned long long at = 0;
    if (lane == 0 && (live & (n == kTile ? 0xffffffffu : (1u << n) - 1u)))
      at = atomicAdd(P.counters, (unsigned long long)__popc(live & (n == kTile ? 0xffffffffu : (1u << n) - 1u)));
    at = __shfl_sync(0xffffffffu, at, 0);
    if (lane < n) {
      if ((live >> lane) & 1u) {
        P.queue[at + __popc(live & ((1u << lane) - 1u))] = (int32_t)(t0 + lane);
      } else {
        const int64_t T = P.tile0 + t0 + lane;
        for (int j = 0; j < JB.n_jobs; ++j) {
          P.mask_u[(size_t)j * P.n_tiles_total + T] = 0u;
          P.mask_q[(size_t)j * P.n_tiles_total + T] = 0u;
        }
      }
    }
  }
}

// The B plane words of group g at one site (col: the population's first pair of the tile, as
// words, plus 2 * site).  Word w of a group sits in pair w >> 1, half w & 1, as in count_wide.
template <int BMAX>
__device__ __forceinline__ void group_words(const uint32_t* col, int g, int B, uint32_t (&x)[BMAX]) {
  if (BMAX == 2) {
    const uint2 v = ld_stream(reinterpret_cast<const uint2*>(col + (size_t)g * 2 * kTile));
    x[0] = v.x;
    x[1] = v.y;
  } else {
#pragma unroll
    for (int b = 0; b < BMAX; ++b) {
      const int w = g * B + b;
      if (b < B) x[b] = __ldg(col + (size_t)(w >> 1) * 2 * kTile + (w & 1));
    }
  }
}

// (num, called) of population L at the sites of a batch in lo:hi (bit 32 g + s = site s of tile g,
// whose index lane g holds in my_tile), stored into those sites' slots of the shared counts.  Lanes
// stride over the population's groups; the counts are those of count_wide, summed over the warp:
//   num = sum_b popc(w_b) << b - (2^B - 1) popc(AND_b w_b),   missing = popc(AND_b w_b)
// ROUND items and two groups per lane at a time, all their loads issued before any sum (a word
// not loaded is 0 and adds nothing).  BMAX == 2 for 2-plane populations (one 8-byte load per
// group), 8 for any other width.
template <int BMAX, int ROUND>
__device__ __noinline__ void gather_sites(const sai_pop_layout& L, const uint32_t* packed, int64_t my_tile,
                                          int64_t pps, uint64_t lo, uint64_t hi, int* s_pop, int per_tile, int n_pops,
                                          int lane) {
  const int B = BMAX == 2 ? 2 : L.bits, G = L.n_groups;
  while (lo | hi) {
    const uint32_t* col[ROUND];  // the item's population column at its site
    int item[ROUND];             // 32 tile + site, -1: none
#pragma unroll
    for (int i = 0; i < ROUND; ++i) {
      item[i] = -1;
      if (lo) {
        item[i] = __ffsll((long long)lo) - 1;
        lo &= lo - 1;
      } else if (hi) {
        item[i] = 64 + __ffsll((long long)hi) - 1;
        hi &= hi - 1;
      }
      const int it = item[i] < 0 ? item[0] : item[i];  // an empty slot loads nothing
      const int64_t T = __shfl_sync(0xffffffffu, (long long)my_tile, it >> 5);
      col[i] = packed + ((size_t)T * pps + L.pair_off) * 2 * kTile + 2 * (it & 31);
    }
    int num[ROUND], miss[ROUND];
#pragma unroll
    for (int i = 0; i < ROUND; ++i) num[i] = miss[i] = 0;
    for (int g = lane; g < G; g += 64) {
      uint32_t x[2][ROUND][BMAX];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
#pragma unroll
        for (int i = 0; i < ROUND; ++i) {
#pragma unroll
          for (int b = 0; b < BMAX; ++b) x[h][i][b] = 0u;
          if (item[i] >= 0 && g + 32 * h < G) group_words<BMAX>(col[i], g + 32 * h, B, x[h][i]);
        }
      }
#pragma unroll
      for (int h = 0; h < 2; ++h) {
#pragma unroll
        for (int i = 0; i < ROUND; ++i) {
          uint32_t andw = 0xffffffffu;
          int s = 0;
#pragma unroll
          for (int b = 0; b < BMAX; ++b) {
            if (b < B) {
              s += __popc(x[h][i][b]) << b;
              andw &= x[h][i][b];
            }
          }
          const int m = __popc(andw);
          num[i] += s - ((1 << B) - 1) * m;
          miss[i] += m;
        }
      }
    }
#pragma unroll
    for (int i = 0; i < ROUND; ++i) {
      if (item[i] < 0) continue;
      const int n = __reduce_add_sync(0xffffffffu, num[i]);
      const int m = __reduce_add_sync(0xffffffffu, miss[i]);
      if (lane == (item[i] & 31)) {
        int* slot = s_pop + (item[i] >> 5) * per_tile + lane;
        slot[0] = n;
        slot[n_pops * kTile] = G * 32 - m;
      }
    }
  }
}

// Phase B: the three stages over batches of batch_tiles queued tiles.  Lane g holds the index of
// the batch's tile g; the next batch's entries are loaded while this batch's stages 2 and 3 run.
__global__ void __launch_bounds__(kSiteWarps * 32, 4)
    k_site_live(const __grid_constant__ SiteParams P, const __grid_constant__ JobBlock JB,
                const __grid_constant__ JobFastBlock JF) {
  extern __shared__ int s_counts[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_pops = P.lay.n_pops, G = P.batch_tiles;
  const int per_tile = 2 * n_pops * kTile;
  int* s_warp = s_counts + warp * G * per_tile;
  const int64_t pps = P.lay.pairs_per_site;
  const int64_t n_live = (int64_t)P.counters[0];
  const int64_t n_batches = (n_live + G - 1) / G;
  // lane 0 claims; the claim of the next batch is in flight while this one is read
  auto claim = [&]() { return lane == 0 ? atomicAdd(P.counters + 1, 1ull) : 0ull; };
  auto tiles_of = [&](int64_t b) {  // lane g: tile g of batch b (lanes past its end repeat its first)
    const int64_t e = b * G + lane;
    return P.tile0 + P.queue[lane < G && e < n_live ? e : b * G];
  };
  int64_t b = (int64_t)__shfl_sync(0xffffffffu, claim(), 0);
  int64_t my_tile = b < n_batches ? tiles_of(b) : 0;
  while (b < n_batches) {
    const unsigned long long claimed = claim();
    const int n = (int)(n_live - b * G < G ? n_live - b * G : G);
    auto tile_at = [&](int g) {  // tile g's first pair at this lane's site
      return P.packed + (size_t)__shfl_sync(0xffffffffu, (long long)my_tile, g) * pps * kTile + lane;
    };

    count_sources<kGateTiles>(P, n, tile_at, s_warp, per_tile, lane);
    const int64_t next_b = (int64_t)__shfl_sync(0xffffffffu, claimed, 0);
    const int64_t next_tile = next_b < n_batches ? tiles_of(next_b) : 0;

    // Stages 2 and 3 run over the whole batch.  Per lane, bits 8 g + j of gate / still: job j's
    // source gate / source and reference gates hold at this lane's site of tile g (SAI_MAX_JOBS
    // == 8).  The counts of a population are valid at the sites it was read for: the source
    // populations at every site, a population read in stage 2 at the sites where any job's source
    // gate holds, one read in stage 3 where any job's reference gate holds too.  Every later use
    // is within that set -- stage 3 sites are a subset of stage 2 sites, and the flags of job j
    // are kept only where both its gates hold -- so a population needed by several stages or jobs
    // is read once, by the first stage that needs it.
    auto num_of_tile = [&](int g) {
      return [=](int pop) { return s_warp[g * per_tile + pop * kTile + lane]; };
    };
    auto called_of_tile = [&](int g) {
      return [=](int pop) { return s_warp[g * per_tile + (n_pops + pop) * kTile + lane]; };
    };
    auto pops_of = [&](uint32_t jobs, bool ref) {
      uint32_t pops = 0;
      for (; jobs; jobs &= jobs - 1) {
        const sai_job& J = JB.job[__ffs(jobs) - 1];
        pops |= 1u << (ref ? J.ref_pop : J.tgt_pop);
      }
      return pops;
    };
    // the sites of tile g where some job of lane_jobs is live
    auto sites_of = [&](uint32_t lane_jobs, int g) {
      return __ballot_sync(0xffffffffu, (lane_jobs >> (8 * g)) & 0xffu);
    };
    // reads population p of tile g for every bit 16 g + p of need (SAI_MAX_POPS == 16) at the sites
    // of tile g where some job of lane_jobs is live: a tile with more than kGatherSites such sites
    // whole, population after population; the others gathered, population by population across
    // the batch
    auto read_stage = [&](uint64_t need, uint32_t lane_jobs) {
      for (int g = 0; g < n; ++g) {
        if (__popc(sites_of(lane_jobs, g)) <= kGatherSites) continue;
        for (uint32_t m = (uint32_t)(need >> (16 * g)) & 0xffffu; m; m &= m - 1) {
          const int pi = __ffs(m) - 1;
          const sai_pop_layout& L = P.lay.pop[pi];
          int* s_num = s_warp + g * per_tile + pi * kTile + lane;
          count_pop<0>(L, tile_at(g) + (size_t)L.pair_off * kTile, s_num[0], s_num[n_pops * kTile]);
        }
        need &= ~(0xffffull << (16 * g));
      }
      uint32_t any = 0;
      for (uint64_t m = need; m; m >>= 16) any |= (uint32_t)m & 0xffffu;
      for (; any; any &= any - 1) {
        const int pi = __ffs(any) - 1;
        uint64_t lo = 0, hi = 0;  // gathered sites, bit 32 g + s (tiles 0, 1 | 2, 3)
        for (int g = 0; g < n; ++g)
          if ((need >> (16 * g + pi)) & 1u) (g < 2 ? lo : hi) |= (uint64_t)sites_of(lane_jobs, g) << (32 * (g & 1));
        const sai_pop_layout& L = P.lay.pop[pi];
        const uint32_t* words = reinterpret_cast<const uint32_t*>(P.packed);
        if (L.bits == 2)
          gather_sites<2, 2>(L, words, my_tile, pps, lo, hi, s_warp + pi * kTile, per_tile, n_pops, lane);
        else
          gather_sites<8, 1>(L, words, my_tile, pps, lo, hi, s_warp + pi * kTile, per_tile, n_pops, lane);
      }
    };

    uint32_t gate = 0;
    for (int g = 0; g < n; ++g) {
      for (int j = 0; j < JB.n_jobs; ++j) {
        bool u, q;
        site_gate(JF.job[j], JB.job[j], P.lay, false, num_of_tile(g), called_of_tile(g), u, q);
        gate |= (uint32_t)(u || q) << (8 * g + j);
      }
    }
    // stage 2: the references of the jobs live on each tile, then the reference gate.  A tile read
    // whole reads the targets of those jobs with them: on a dense tile they are needed almost
    // always, and one stage of whole-tile reads keeps the all-live case close to one pass (DESIGN 4).
    const uint32_t live1 = __reduce_or_sync(0xffffffffu, gate);
    uint64_t need2 = 0;
    for (int g = 0; g < n; ++g) {
      const uint32_t jobs = (live1 >> (8 * g)) & 0xffu;
      uint32_t pops = pops_of(jobs, true);
      if (__popc(sites_of(gate, g)) > kGatherSites) pops |= pops_of(jobs, false);
      need2 |= (uint64_t)(pops & ~P.gate_pops) << (16 * g);
    }
    read_stage(need2, gate);
    uint32_t still = 0;
    for (uint32_t m = live1; m; m &= m - 1) {
      const int g = (__ffs(m) - 1) >> 3, j = (__ffs(m) - 1) & 7;
      bool u, q;
      site_gate(JF.job[j], JB.job[j], P.lay, true, num_of_tile(g), called_of_tile(g), u, q);
      still |= (uint32_t)(u || q) << (8 * g + j);
    }
    // stage 3: the targets of the jobs still live
    const uint32_t live2 = __reduce_or_sync(0xffffffffu, still);
    uint64_t need3 = 0;
    for (int g = 0; g < n; ++g)
      need3 |= (uint64_t)(pops_of((live2 >> (8 * g)) & 0xffu, false) & ~P.gate_pops) << (16 * g);
    read_stage(need3 & ~need2, still);

    for (int g = 0; g < n; ++g) {
      const int64_t T = __shfl_sync(0xffffffffu, (long long)my_tile, g);
      const int64_t site = T * kTile + lane;
      for (int j = 0; j < JB.n_jobs; ++j) {
        const int bit = 8 * g + j;
        uint32_t mu = 0, mq = 0;
        if ((live2 >> bit) & 1u) {
          // lanes where job j's gates fail may hold counts never read for this tile: they are
          // evaluated as fully called sites with a count of 0 (so they keep the warp on the
          // integer path) and their flags dropped
          const bool mine = (still >> bit) & 1u;
          const SiteFlags f = eval_site_fast(
              JF.job[j], JB.job[j], P.lay, [&](int pop) { return mine ? num_of_tile(g)(pop) : 0; },
              [&](int pop) { return mine ? called_of_tile(g)(pop) : P.lay.pop[pop].n_samples; });
          mu = __ballot_sync(0xffffffffu, f.u && mine);
          mq = __ballot_sync(0xffffffffu, f.q && mine);
          if (f.q && mine) P.qval[(size_t)j * P.qval_stride + site] = f.q_tgt_freq;
        }
        if (lane == 0) {
          P.mask_u[(size_t)j * P.n_tiles_total + T] = mu;
          P.mask_q[(size_t)j * P.n_tiles_total + T] = mq;
        }
      }
    }
    b = next_b;
    my_tile = next_tile;
  }
}

struct CountFlagParams {
  sai_layout lay;
  const int32_t* num;
  const int32_t* called;
  int64_t count_stride;
  int64_t n_sites;
  uint32_t* mask_u;
  uint32_t* mask_q;
  double* qval;
  int64_t qval_stride;
  int64_t n_tiles_total;
};

// Site conditions from cached counts (threshold sweeps, BASELINE config 5): lane == site, one warp
// takes kFcTiles consecutive tiles per trip.  The counts of every population are loaded ONCE --
// 2 * NP * kFcTiles independent coalesced 128-byte loads in flight per warp -- and then all jobs
// of the launch (up to 8 parameter sets) are evaluated out of registers, so a set costs 1/8 of the
// count traffic (8 (2 + K) bytes per site, L2-resident for chromosome-scale inputs) plus ~50
// integer instructions per site.  NP = populations of the layout held in registers (1..4);
// NP == 0 is the generic version that re-reads the counts per job through L1.
constexpr int kFcTiles = 4;

template <int NP>
__device__ __forceinline__ int pick(const int (&a)[NP > 0 ? NP : 1], int pop) {
  int r = a[0];
#pragma unroll
  for (int i = 1; i < NP; ++i) r = pop == i ? a[i] : r;  // pop is warp-uniform (kernel parameter)
  return r;
}

template <int NP>
__global__ void __launch_bounds__(256)
    k_flags_from_counts(const __grid_constant__ CountFlagParams P, const __grid_constant__ JobBlock JB,
                        const __grid_constant__ JobFastBlock JF) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t n_trips = (P.n_tiles_total + kFcTiles - 1) / kFcTiles;
  for (int64_t trip = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; trip < n_trips; trip += warps) {
    const int64_t T0 = trip * kFcTiles;
    int num[kFcTiles][NP > 0 ? NP : 1], cal[kFcTiles][NP > 0 ? NP : 1];
    if (NP > 0) {
#pragma unroll
      for (int t = 0; t < kFcTiles; ++t) {
        const int64_t site = (T0 + t) * kTile + lane;
        const bool live = site < P.n_sites;
#pragma unroll
        for (int p = 0; p < NP; ++p) {
          num[t][p] = live ? __ldg(P.num + (size_t)p * P.count_stride + site) : 0;
          cal[t][p] = live ? __ldg(P.called + (size_t)p * P.count_stride + site) : 0;
        }
      }
    }
    for (int j = 0; j < JB.n_jobs; ++j) {
      const sai_job& J = JB.job[j];
      uint32_t mu[kFcTiles], mq[kFcTiles];
#pragma unroll
      for (int t = 0; t < kFcTiles; ++t) {
        const int64_t site = (T0 + t) * kTile + lane;
        const bool live = site < P.n_sites;
        SiteFlags f;
        if (NP > 0) {
          f = eval_site_fast(JF.job[j], J, P.lay, [&](int pop) { return pick<NP>(num[t], pop); },
                             [&](int pop) { return pick<NP>(cal[t], pop); });
        } else {
          f = eval_site_fast(
              JF.job[j], J, P.lay,
              [&](int pop) { return live ? __ldg(P.num + (size_t)pop * P.count_stride + site) : 0; },
              [&](int pop) { return live ? __ldg(P.called + (size_t)pop * P.count_stride + site) : 0; });
        }
        mu[t] = __ballot_sync(0xffffffffu, f.u);
        mq[t] = __ballot_sync(0xffffffffu, f.q);
        if (f.q) P.qval[(size_t)j * P.qval_stride + site] = f.q_tgt_freq;
      }
      // lanes 0..3 store the trip's four mask words side by side (one 16-byte segment per array)
      uint32_t wu = mu[0], wq = mq[0];
#pragma unroll
      for (int t = 1; t < kFcTiles; ++t) {
        wu = lane == t ? mu[t] : wu;
        wq = lane == t ? mq[t] : wq;
      }
      if (lane < kFcTiles && T0 + lane < P.n_tiles_total) {
        P.mask_u[(size_t)j * P.n_tiles_total + T0 + lane] = wu;
        P.mask_q[(size_t)j * P.n_tiles_total + T0 + lane] = wq;
      }
    }
  }
}

static void fill_job_fast(const sai_layout& lay, const JobBlock& JB, JobFastBlock& JF) {
  memset(&JF, 0, sizeof(JF));
  for (int j = 0; j < JB.n_jobs; ++j) build_job_fast(lay, JB.job[j], JF.job[j]);
}

template <int MODE, bool FUSED>
static int launch_site(const SiteParams& P, const JobBlock& JB, cudaStream_t st) {
  if (P.n_tiles == 0) return SAI_OK;
  const size_t smem = (size_t)kSiteWarps * 2 * P.lay.n_pops * kTile * sizeof(int);
  int occ = 0;
  SAI_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_site<MODE, FUSED>,
                                                               kSiteWarps * 32, smem));
  if (occ < 1) occ = 1;
  int64_t want = (P.n_tiles + kSiteWarps - 1) / kSiteWarps;
  int64_t cap = (int64_t)sm_count() * occ;
  int grid = (int)(want < cap ? want : cap);
  JobFastBlock JF;
  fill_job_fast(P.lay, JB, JF);
  k_site<MODE, FUSED><<<grid, kSiteWarps * 32, smem, st>>>(P, JB, JF);
  SAI_CUDA_CHECK(cudaGetLastError());
  return SAI_OK;
}

static int launch_site_gated(SiteParams P, const JobBlock& JB, cudaStream_t st) {
  if (P.n_tiles == 0) return SAI_OK;
  SAI_REQUIRE(P.n_tiles <= INT32_MAX, "too many tiles for one genotype pass (%lld)", (long long)P.n_tiles);
  P.gate_pops = 0;
  for (int j = 0; j < JB.n_jobs; ++j) {
    const sai_job& J = JB.job[j];
    if (J.u.enabled || J.q.enabled)
      for (int k = 0; k < J.n_src; ++k) P.gate_pops |= 1u << J.src_pop[k];
  }
  JobFastBlock JF;
  fill_job_fast(P.lay, JB, JF);
  P.scan_pops = 0;
  P.scan_all = 0;
  P.n_scan = 0;
  bool wide = false;
  for (int j = 0; j < JB.n_jobs; ++j) {
    const sai_job& J = JB.job[j];
    const JobFast& F = JF.job[j];
    if (!(J.u.enabled || J.q.enabled)) continue;
    if (!F.ok) {  // no integer intervals: the gate is decided by divisions only
      P.scan_all = 1;
      continue;
    }
    ScanTest& T = P.scan[P.n_scan++];
    T.pop = J.src_pop[0];
    T.den = F.den_src[0];
    T.n = 0;
    const CondFast* cf[2] = {&F.u, &F.q};
    const bool en[2] = {J.u.enabled != 0, J.q.enabled != 0};
    for (int c = 0; c < 2; ++c) {
      if (!en[c]) continue;
      T.lo[T.n] = cf[c]->y_lo[0], T.hi[T.n++] = cf[c]->y_hi[0];
      if (!J.anc_allele_available) T.lo[T.n] = cf[c]->f_lo[0], T.hi[T.n++] = cf[c]->f_hi[0];
    }
    P.scan_pops |= 1u << T.pop;
    wide = wide || P.lay.pop[T.pop].bits != 2;
  }
  const int tile_bytes = 2 * P.lay.n_pops * kTile * (int)sizeof(int);
  P.batch_tiles = std::max(1, std::min(kGateTiles, kGateSmemPerWarp / tile_bytes));
  const size_t smem_live = (size_t)kSiteWarps * P.batch_tiles * tile_bytes;
  auto scan = wide ? k_site_scan<true> : k_site_scan<false>;
  int occ_scan = 0, occ_live = 0;
  SAI_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_scan, scan, kSiteWarps * 32, 0));
  SAI_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_live, k_site_live, kSiteWarps * 32, smem_live));
  const int64_t want_scan = (P.n_tiles + kSiteWarps * kTile - 1) / (kSiteWarps * kTile);
  const int64_t want_live = ((P.n_tiles + P.batch_tiles - 1) / P.batch_tiles + kSiteWarps - 1) / kSiteWarps;
  const int64_t cap_scan = (int64_t)sm_count() * std::max(occ_scan, 1);
  const int64_t cap_live = (int64_t)sm_count() * std::max(occ_live, 1);
  // counters, then the queue
  void* scratch = nullptr;
  if (int rc = scratch_alloc(&scratch, 2 * sizeof(unsigned long long) + (size_t)P.n_tiles * sizeof(int32_t), st))
    return rc;
  P.counters = static_cast<unsigned long long*>(scratch);
  P.queue = reinterpret_cast<int32_t*>(P.counters + 2);
  SAI_CUDA_CHECK(cudaMemsetAsync(scratch, 0, 2 * sizeof(unsigned long long), st));
  scan<<<(int)std::min(want_scan, cap_scan), kSiteWarps * 32, 0, st>>>(P, JB);
  SAI_CUDA_CHECK(cudaGetLastError());
  k_site_live<<<(int)std::min(want_live, cap_live), kSiteWarps * 32, smem_live, st>>>(P, JB, JF);
  SAI_CUDA_CHECK(cudaGetLastError());
  return scratch_free(scratch, st);
}


#ifdef SAI_EXPERIMENTS
// Batch table shared by the experimental variants: the tile's pairs cut into batches of up
// to 8 pairs that never straddle a population (pair index | valid-1 | population | last-of-population).
__device__ __forceinline__ uint32_t batch_entry(int pair, int valid, int pop, bool last) {
  return (uint32_t)pair | ((uint32_t)(valid - 1) << 20) | ((uint32_t)pop << 23) | ((uint32_t)last << 27);
}

// ---------------------------------------------------------------------------
// Variants 5-7: bulk-copy ring (experiment, measured slower than variant 0 --
// profiles/round1_notes.md).  Batches of up to 8 pairs are fetched by the copy
// engine (cp.async.bulk global -> shared, completion on an mbarrier) into a
// per-warp ring of STAGES 2 KB buffers, so the bytes in flight are bounded by
// shared memory (up to ~190 KB per SM) instead of by registers, and the adder
// tree / epilogue never drain the memory pipe.  lane == site: every lane reads
// its own 8-byte pair of each row, conflict-free.
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tWAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

template <bool FUSED, int STAGES, int MINB>
__global__ void __launch_bounds__(kSiteWarps * 32, MINB)
    k_site_ring(const __grid_constant__ SiteParams P, const __grid_constant__ JobBlock JB,
                const __grid_constant__ JobFastBlock JF, int n_batches, int tab_words) {
  extern __shared__ __align__(128) unsigned char s_raw[];
  // [ring: warps x STAGES x 2 KB][mbarriers: warps x STAGES x 8 B][table][counts]
  uint2* s_ring = reinterpret_cast<uint2*>(s_raw);
  unsigned long long* s_bar = reinterpret_cast<unsigned long long*>(s_raw + (size_t)kSiteWarps * STAGES * 2048);
  uint32_t* s_tab = reinterpret_cast<uint32_t*>(s_bar + kSiteWarps * STAGES);
  int* s_counts = reinterpret_cast<int*>(s_tab + tab_words);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_pops = P.lay.n_pops;
  if (threadIdx.x == 0) {
    int b = 0;
    for (int pi = 0; pi < n_pops; ++pi) {
      const sai_pop_layout& L = P.lay.pop[pi];
      for (int q = 0; q < L.n_pairs; q += 8) {
        const int valid = L.n_pairs - q < 8 ? L.n_pairs - q : 8;
        s_tab[b++] = batch_entry(L.pair_off + q, valid, pi, q + 8 >= L.n_pairs);
      }
    }
  }
  if (lane == 0) {
    for (int st = 0; st < STAGES; ++st) mbar_init(smem_u32(s_bar + warp * STAGES + st), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  int* s_num = s_counts + warp * (2 * n_pops * kTile);
  int* s_cal = s_num + n_pops * kTile;
  const int64_t pps = P.lay.pairs_per_site;
  const int64_t stride = (int64_t)gridDim.x * kSiteWarps;
  int64_t t = (int64_t)blockIdx.x * kSiteWarps + warp;
  if (t >= P.n_tiles) return;
  const uint2* my_ring = s_ring + (size_t)warp * STAGES * 256;
  const uint32_t ring0 = smem_u32(my_ring), bar0 = smem_u32(s_bar + warp * STAGES);
  const unsigned char* base = reinterpret_cast<const unsigned char*>(P.packed) + (size_t)P.tile0 * pps * 256;

  // producer cursor (lane 0): the next chunk to request
  int64_t pt = t;
  int pb = 0;
  auto issue = [&](int st) {  // lane 0 only; returns with the cursor advanced
    if (pt >= P.n_tiles) return;
    const uint32_t e = s_tab[pb];
    const uint32_t bytes = (((e >> 20) & 7u) + 1u) * 256u;
    const uint32_t bar = bar0 + 8u * st;
    mbar_expect_tx(bar, bytes);
    bulk_g2s(ring0 + 2048u * st, base + ((size_t)pt * pps + (e & 0xfffffu)) * 256, bytes, bar);
    if (++pb == n_batches) {
      pb = 0;
      pt += stride;
    }
  };
  if (lane == 0)
    for (int st = 0; st < STAGES; ++st) issue(st);

  SliceCounter ca, cb, cm;
  int b = 0, st = 0;
  uint32_t parity = 0;
  while (t < P.n_tiles) {
    const uint32_t e = s_tab[b];
    const int valid = (int)((e >> 20) & 7u) + 1;
    mbar_wait(bar0 + 8u * st, parity);
    const uint2* buf = my_ring + st * 256 + lane;
    uint32_t a[8], bb[8], m[8];
    uint32_t mo = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const uint2 v = buf[i * kTile];
      const uint32_t keep = i < valid ? 0xffffffffu : 0u;  // rows beyond the batch hold stale bytes
      a[i] = v.x & keep;
      bb[i] = v.y & keep;
      m[i] = a[i] & bb[i];
      mo |= m[i];
    }
    // every lane has its rows in registers (the vote needs them): the stage can be refilled
    const bool any_missing = __any_sync(0xffffffffu, mo != 0u);
    if (lane == 0) issue(st);
    ca.add8(a);
    cb.add8(bb);
    if (any_missing) cm.add8(m);
    if (e >> 27) {  // last batch of its population
      const int pi = (int)((e >> 23) & 15u);
      const int miss = cm.total();
      const int num = ca.total() + 2 * cb.total() - 3 * miss;
      const int called = P.lay.pop[pi].n_groups * 32 - miss;
      s_num[pi * kTile + lane] = num;
      s_cal[pi * kTile + lane] = called;
      if (P.num) {
        const int64_t site = (P.tile0 + t) * kTile + lane;
        P.num[(size_t)pi * P.count_stride + site] = num;
        P.called[(size_t)pi * P.count_stride + site] = called;
      }
      ca = SliceCounter();
      cb = SliceCounter();
      cm = SliceCounter();
    }
    if (++st == STAGES) {
      st = 0;
      parity ^= 1u;
    }
    if (++b == n_batches) {
      if (FUSED) {
        const int64_t T = P.tile0 + t;
        const int64_t site = T * kTile + lane;
        for (int j = 0; j < JB.n_jobs; ++j) {
          const sai_job& J = JB.job[j];
          SiteFlags f = eval_site_fast(
              JF.job[j], J, P.lay, [&](int pop) { return s_num[pop * kTile + lane]; },
              [&](int pop) { return s_cal[pop * kTile + lane]; });
          const uint32_t mu = __ballot_sync(0xffffffffu, f.u);
          const uint32_t mq = __ballot_sync(0xffffffffu, f.q);
          if (lane == 0) {
            P.mask_u[(size_t)j * P.n_tiles_total + T] = mu;
            P.mask_q[(size_t)j * P.n_tiles_total + T] = mq;
          }
          if (f.q) P.qval[(size_t)j * P.qval_stride + site] = f.q_tgt_freq;
        }
      }
      b = 0;
      t += stride;
    }
  }
}

template <bool FUSED, int STAGES, int MINB>
static int launch_site_ring(const SiteParams& P, const JobBlock& JB, cudaStream_t st) {
  if (P.n_tiles == 0) return SAI_OK;
  int n_batches = 0;
  for (int p = 0; p < P.lay.n_pops; ++p) n_batches += (P.lay.pop[p].n_pairs + 7) / 8;
  const int tab_words = (n_batches + 31) & ~31;
  const size_t smem = (size_t)kSiteWarps * STAGES * (2048 + 8) +
                      sizeof(int) * ((size_t)tab_words + (size_t)kSiteWarps * 2 * P.lay.n_pops * kTile);
  auto kern = k_site_ring<FUSED, STAGES, MINB>;
  if (smem > 227 * 1024) return -1000;  // caller falls back
  SAI_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 0;
  SAI_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kSiteWarps * 32, smem));
  if (occ < 1) occ = 1;
  const int64_t want = (P.n_tiles + kSiteWarps - 1) / kSiteWarps;
  const int64_t cap = (int64_t)sm_count() * occ;
  JobFastBlock JF;
  fill_job_fast(P.lay, JB, JF);
  kern<<<(int)(want < cap ? want : cap), kSiteWarps * 32, smem, st>>>(P, JB, JF, n_batches, tab_words);
  SAI_CUDA_CHECK(cudaGetLastError());
  return SAI_OK;
}

static bool all_two_planes(const sai_layout& lay) {
  for (int p = 0; p < lay.n_pops; ++p)
    if (lay.pop[p].bits != 2) return false;
  return true;
}

#endif  // SAI_EXPERIMENTS

}  // namespace sai

using namespace sai;

extern "C" {

int sai_site_counts(const sai_layout* lay, const void* d_packed, int64_t tile0, int64_t n_tiles,
                    int32_t* d_num, int32_t* d_called, int64_t stride, int32_t variant,
                    void* stream) {
  if (int rc = validate_layout(lay)) return rc;
  SAI_REQUIRE(d_packed && d_num && d_called, "NULL device pointer");
  SAI_REQUIRE(tile0 >= 0 && n_tiles >= 0 && stride >= (tile0 + n_tiles) * kTile, "bad tile range / stride");
  SiteParams P{};
  P.lay = *lay;
  P.packed = static_cast<const uint2*>(d_packed);
  P.tile0 = tile0;
  P.n_tiles = n_tiles;
  P.n_tiles_total = tile0 + n_tiles;
  P.num = d_num;
  P.called = d_called;
  P.count_stride = stride;
  JobBlock JB{};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
#ifdef SAI_EXPERIMENTS
  if (variant >= 5 && variant <= 7 && all_two_planes(*lay)) {
    const int rc = variant == 5   ? launch_site_ring<false, 3, 4>(P, JB, st)
                   : variant == 6 ? launch_site_ring<false, 4, 3>(P, JB, st)
                                  : launch_site_ring<false, 6, 2>(P, JB, st);
    if (rc != -1000) return rc;
  }
  if (variant == 2) return launch_site<2, false>(P, JB, st);
  if (variant == 1) return launch_site<1, false>(P, JB, st);
#else
  SAI_REQUIRE(variant == 0, "variant %d exists only in -DSAI_EXPERIMENTS builds", variant);
#endif
  return launch_site<0, false>(P, JB, st);
}

int sai_site_flags(const sai_layout* lay, const void* d_packed, int64_t tile0, int64_t n_tiles,
                   int64_t n_tiles_total, const sai_job* jobs, int32_t n_jobs, uint32_t* d_mask_u,
                   uint32_t* d_mask_q, double* d_qval, int64_t qval_stride, int32_t* d_num,
                   int32_t* d_called, int64_t count_stride, int32_t variant, void* stream) {
  if (int rc = validate_layout(lay)) return rc;
  if (int rc = validate_jobs(lay, jobs, n_jobs)) return rc;
  SAI_REQUIRE(d_packed && d_mask_u && d_mask_q && d_qval, "NULL device pointer");
  SAI_REQUIRE(tile0 >= 0 && n_tiles >= 0 && tile0 + n_tiles <= n_tiles_total, "bad tile range");
  SAI_REQUIRE(qval_stride >= n_tiles_total * kTile, "qval_stride too small");
  SAI_REQUIRE((d_num == nullptr) == (d_called == nullptr), "d_num/d_called must both be set or NULL");
  SAI_REQUIRE(!d_num || count_stride >= n_tiles_total * kTile, "count_stride too small");
  SiteParams P{};
  P.lay = *lay;
  P.packed = static_cast<const uint2*>(d_packed);
  P.tile0 = tile0;
  P.n_tiles = n_tiles;
  P.n_tiles_total = n_tiles_total;
  P.mask_u = d_mask_u;
  P.mask_q = d_mask_q;
  P.qval = d_qval;
  P.qval_stride = qval_stride;
  P.num = d_num;
  P.called = d_called;
  P.count_stride = count_stride;
  JobBlock JB{};
  JB.n_jobs = n_jobs;
  for (int j = 0; j < n_jobs; ++j) JB.job[j] = jobs[j];
  cudaStream_t st = static_cast<cudaStream_t>(stream);
#ifdef SAI_EXPERIMENTS
  if (variant >= 5 && variant <= 7 && all_two_planes(*lay)) {
    const int rc = variant == 5   ? launch_site_ring<true, 3, 4>(P, JB, st)
                   : variant == 6 ? launch_site_ring<true, 4, 3>(P, JB, st)
                                  : launch_site_ring<true, 6, 2>(P, JB, st);
    if (rc != -1000) return rc;
  }
  if (variant == 2) return launch_site<2, true>(P, JB, st);
  if (variant == 1) return launch_site<1, true>(P, JB, st);
#else
  SAI_REQUIRE(variant == 0, "variant %d exists only in -DSAI_EXPERIMENTS builds", variant);
#endif
  // stored counts: every population is read anyway
  if (d_num) return launch_site<0, true>(P, JB, st);
  return launch_site_gated(P, JB, st);
}

int sai_flags_from_counts(const sai_layout* lay, const int32_t* d_num, const int32_t* d_called,
                          int64_t count_stride, int64_t n_sites, const sai_job* jobs,
                          int32_t n_jobs, uint32_t* d_mask_u, uint32_t* d_mask_q, double* d_qval,
                          int64_t qval_stride, void* stream) {
  if (int rc = validate_layout(lay)) return rc;
  if (int rc = validate_jobs(lay, jobs, n_jobs)) return rc;
  SAI_REQUIRE(d_num && d_called && d_mask_u && d_mask_q && d_qval, "NULL device pointer");
  SAI_REQUIRE(n_sites >= 0 && count_stride >= n_sites && qval_stride >= n_sites, "bad strides");
  if (n_sites == 0) return SAI_OK;
  CountFlagParams P{};
  P.lay = *lay;
  P.num = d_num;
  P.called = d_called;
  P.count_stride = count_stride;
  P.n_sites = n_sites;
  P.mask_u = d_mask_u;
  P.mask_q = d_mask_q;
  P.qval = d_qval;
  P.qval_stride = qval_stride;
  P.n_tiles_total = sai_num_tiles(n_sites);
  JobBlock JB{};
  JB.n_jobs = n_jobs;
  for (int j = 0; j < n_jobs; ++j) JB.job[j] = jobs[j];
  const int64_t n_trips = (P.n_tiles_total + kFcTiles - 1) / kFcTiles;
  const int64_t want = (n_trips + 7) / 8;  // 8 warps per block
  const int64_t cap = (int64_t)sm_count() * 16;
  const int grid = (int)(want < cap ? want : cap);
  JobFastBlock JF;
  fill_job_fast(*lay, JB, JF);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (lay->n_pops) {
    case 1: k_flags_from_counts<1><<<grid, 256, 0, st>>>(P, JB, JF); break;
    case 2: k_flags_from_counts<2><<<grid, 256, 0, st>>>(P, JB, JF); break;
    case 3: k_flags_from_counts<3><<<grid, 256, 0, st>>>(P, JB, JF); break;
    case 4: k_flags_from_counts<4><<<grid, 256, 0, st>>>(P, JB, JF); break;
    default: k_flags_from_counts<0><<<grid, 256, 0, st>>>(P, JB, JF); break;
  }
  SAI_CUDA_CHECK(cudaGetLastError());
  return SAI_OK;
}

}  // extern "C"
