// N4: the DD statistic (sai/stats/dd_statistic.py:62-77).
//
// Reference, per window and source population k with individuals a = 0..m-1:
//     seq_divs_src_ref[a, j] = sum_sites |src[site, a] - ref[site, j]|      (cdist cityblock, :70)
//     mean_src_ref[a]        = mean_j seq_divs_src_ref[a, j]                (:74)
//     dd = mean_a (mean_src_ref[a] - mean_src_tgt[a])                       (:77)
// on the RAW per-individual allele sums: a missing call enters the distance
// with its negative value (-1 for "0/.", -2 for "./." in diploid data).
//
// Everything up to the two means is integer arithmetic, so the kernels return
// the exact integers
//     ref_sum[k][window][a] = sum_j sum_sites |src_a - ref_j|      (tgt_sum likewise)
// and the caller forms  mean_a(ref_sum/n_ref - tgt_sum/n_tgt)  in float64 with
// the reference's own operations (the sums of integers below 2^53 are exact in
// the reference's float64 too), which makes DD bit-exact.
//
// Per site, sum_j |s - ref_j| = sum_u c_u |s - u| + sum_{j not in c} |s - r_j|,
// with c_u the number of individuals holding the called value u (u = 0..14); the rest are the
// missing calls (raw values from the negative-value table) and, in populations of 5-8 planes,
// the *wide* calls (values 15..127, read back from the planes):
//   k_site_hist   one genotype pass over ref and tgt -> c_u per site (bit-plane
//                 match masks + POPC; lane == site as in k_site), plus the number of
//                 wide calls of a 5-8-plane population
//   k_site_dd     per site and source individual the two distances sum_j |src_a - ref_j|,
//                 sum_j |src_a - tgt_j| (called part from c_u, wide calls from the planes,
//                 missing calls from the negative-value table: the bit-planes keep a single
//                 "missing" code, the table restores the raw values) -- once per site, not once
//                 per overlapping window
//   k_window_dd   one warp per (source population, window): exact int64 sums of those
//                 per-site integers over the window's site range.
// The site and entry kernels come in two builds: kMaxB = 4 for layouts of 2-4 planes (the
// common case, unchanged) and kMaxB = 8 as soon as one DD population has 5-8 planes.
#include <algorithm>

#include "common.cuh"
#include "popcount.cuh"
#include "scratch.cuh"

namespace sai {

constexpr int kHistWarps = 8;
constexpr int kDdWarps = 8;
constexpr int kMaxCodes = 15;  // called values of a 4-plane population; histogram rows of values
                               // 0..14 in wider populations, whose row kMaxCodes counts wide calls

// histogram rows holding called values (2^B - 1, or 0..14 when the population is wider)
template <int kMaxB>
__device__ __forceinline__ int value_rows(int bits) {
  return kMaxB > 4 && bits > 4 ? kMaxCodes : (1 << bits) - 1;
}

struct HistParams {
  const uint2* packed;
  int32_t pairs_per_site;
  int32_t n_sites;
  int64_t n_tiles;
  int64_t stride;
  int32_t n_slots;
  int32_t pair_off[SAI_MAX_POPS], n_groups[SAI_MAX_POPS], bits[SAI_MAX_POPS], code_base[SAI_MAX_POPS],
      pad[SAI_MAX_POPS];
  int32_t* hist;
  unsigned long long* missing;  // [n_slots] or NULL
};

__device__ __forceinline__ uint32_t plane_word(const uint2* __restrict__ col, int word) {
  // word `word` of a population column at this lane's site (col already points at pair 0, this site)
  const uint32_t* p = reinterpret_cast<const uint32_t*>(col + (size_t)(word >> 1) * kTile);
  return __ldg(p + (word & 1));
}

__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// grid-stride over tiles, one warp per tile, lane == site
template <int kMaxB>
__global__ void __launch_bounds__(kHistWarps * 32, 4) k_site_hist(const __grid_constant__ HistParams P) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // population by population (each one's pairs are a contiguous 256 B x n_pairs run of a tile)
  for (int q = 0; q < P.n_slots; ++q) {
    unsigned long long miss_total = 0;
    for (int64_t T = (int64_t)blockIdx.x * kHistWarps + warp; T < P.n_tiles; T += (int64_t)gridDim.x * kHistWarps) {
      const uint2* tile = P.packed + (size_t)T * P.pairs_per_site * kTile + lane;
      const int64_t site = T * kTile + lane;
      const uint2* col = tile + (size_t)P.pair_off[q] * kTile;
      const int B = P.bits[q], G = P.n_groups[q];
      int32_t* out = P.hist + (size_t)P.code_base[q] * P.stride + site;
      int miss = 0;
      if (B == 2) {
        // three word streams (value 1, value 2, missing) through carry-save adders, 8 groups per trip
        SliceCounter k1, k2, km;
        int g = 0;
        for (; g + 8 <= G; g += 8) {
          uint2 w[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) w[i] = ld_stream(col + (size_t)(g + i) * kTile);
          uint32_t x1[8], x2[8], xm[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            x1[i] = w[i].x & ~w[i].y;
            x2[i] = w[i].y & ~w[i].x;
            xm[i] = w[i].x & w[i].y;
          }
          k1.add8(x1);
          k2.add8(x2);
          km.add8(xm);
        }
        int c1 = k1.total(), c2 = k2.total();
        miss = km.total();
        for (; g < G; ++g) {
          const uint2 w = ld_stream(col + (size_t)g * kTile);
          c1 += __popc(w.x & ~w.y);
          c2 += __popc(w.y & ~w.x);
          miss += __popc(w.x & w.y);
        }
        out[0] = 32 * G - c1 - c2 - miss;
        out[P.stride] = c1;
        out[2 * P.stride] = c2;
      } else if (kMaxB > 4 && B > 4) {
        // values 0..14 as in a 4-plane population (planes 4.. clear), then one row of wide calls:
        // not all-ones and either a high plane set or value 15 (planes 0..3 set, the rest clear)
        int cnt[kMaxCodes];
#pragma unroll
        for (int u = 0; u < kMaxCodes; ++u) cnt[u] = 0;
        int wide = 0;
        for (int g = 0; g < G; ++g) {
          uint32_t w[4];
#pragma unroll
          for (int b = 0; b < 4; ++b) w[b] = plane_word(col, g * B + b);
          const uint32_t low_ones = w[0] & w[1] & w[2] & w[3];
          uint32_t hi = 0, all = low_ones;
          for (int b = 4; b < B; ++b) {
            const uint32_t x = plane_word(col, g * B + b);
            hi |= x;
            all &= x;
          }
          miss += __popc(all);
          wide += __popc((hi | low_ones) & ~all);
#pragma unroll
          for (int u = 0; u < kMaxCodes; ++u) {
            uint32_t m = ~hi;
#pragma unroll
            for (int b = 0; b < 4; ++b) m &= ((u >> b) & 1) ? w[b] : ~w[b];
            cnt[u] += __popc(m);
          }
        }
#pragma unroll
        for (int u = 0; u < kMaxCodes; ++u) out[(size_t)u * P.stride] = cnt[u];
        out[(size_t)kMaxCodes * P.stride] = wide;
      } else {
        int cnt[kMaxCodes];
#pragma unroll
        for (int u = 0; u < kMaxCodes; ++u) cnt[u] = 0;
        const int n_called = (1 << B) - 1;
        for (int g = 0; g < G; ++g) {
          uint32_t w[4];
#pragma unroll
          for (int b = 0; b < 4; ++b) w[b] = b < B ? plane_word(col, g * B + b) : 0u;
          uint32_t all = 0xffffffffu;
#pragma unroll
          for (int b = 0; b < 4; ++b)
            if (b < B) all &= w[b];
          miss += __popc(all);
#pragma unroll
          for (int u = 0; u < kMaxCodes; ++u) {
            if (u < n_called) {
              uint32_t m = 0xffffffffu;
#pragma unroll
              for (int b = 0; b < 4; ++b)
                if (b < B) m &= ((u >> b) & 1) ? w[b] : ~w[b];
              cnt[u] += __popc(m);
            }
          }
        }
#pragma unroll
        for (int u = 0; u < kMaxCodes; ++u)
          if (u < n_called) out[(size_t)u * P.stride] = cnt[u];
      }
      if (site < P.n_sites) miss_total += miss - P.pad[q];
    }
    // one atomic per warp and population (per tile they would serialise on a single address)
    if (P.missing) {
      const unsigned long long tot = warp_sum_u64(miss_total);
      if (lane == 0 && tot) atomicAdd(P.missing + q, tot);
    }
  }
}

// ---------------------------------------------------------------------------
struct DdPop {
  int32_t pair_off, bits, n_samples, code_base;  // code_base: first histogram row (ref / tgt only)
  int64_t neg_lo, neg_hi;                        // this population's slice of the negative-value table
};

struct DdParams {
  const uint2* packed;
  int32_t pairs_per_site;
  const int32_t* pos;
  int32_t n_sites;
  int64_t n_tiles;
  const int64_t* ws;
  const int64_t* we;
  int32_t W;
  const int32_t* hist;
  int64_t stride;
  DdPop ref, tgt;
  int32_t n_src;
  DdPop src[SAI_MAX_SRC];
  int32_t slot0[SAI_MAX_SRC];  // first row pair of source population k in `dist`
  const int32_t* neg_site;
  const int32_t* neg_ind;
  const int32_t* neg_val;
  int32_t* dist;       // [slot][2][stride]: per site, sum_j |src_a - ref_j| and sum_j |src_a - tgt_j|
  long long* ref_sum;  // [n_src][W][m_max]
  long long* tgt_sum;
  int32_t m_max;
  int32_t* err;  // set to 1 when a missing code has no entry in the negative-value table
};

__device__ __forceinline__ int clamp_k(int64_t k) {
  return k > 2147483647ll ? 2147483647 : (k < -2147483647ll ? -2147483647 : (int)k);
}

// cooperative 32-ary lower bound over a sorted int32 array slice [0, n)
__device__ __forceinline__ int64_t warp_lower_bound(const int32_t* __restrict__ a, int64_t n, int64_t key, int lane) {
  const int k = clamp_k(key);
  int64_t lo = key > 2147483647ll ? n : 0, hi = n;
  while (hi > lo) {
    const int64_t nn = hi - lo;
    const int64_t s = nn > 32 ? (nn + 31) >> 5 : 1;
    const int64_t idx = lo + (lane + 1) * s - 1;
    const bool p = idx < hi && __ldg(a + idx) < k;
    const int c = __popc(__ballot_sync(0xffffffffu, p));
    const int64_t nhi = lo + (c + 1) * s - 1;
    lo += c * s;
    if (nhi < hi) hi = nhi;
    if (lo > hi) lo = hi;
  }
  return lo;
}

// ---- pass 2: per-site distances, once per site -------------------------------------------------
// A site lies in win_len / win_step windows; its contribution
//     dist[a][ref] = sum_j |src_a - ref_j| = sum_u c_u |s_a - u| + sum_{j not in c} |s_a - r_j|
// (s_a: the source individual's called value, or its raw negative value from the table when its
// call is missing) does not depend on the window, so it is computed once and the window kernel
// only adds integers.  Two launches:
//   k_site_dd    site-driven, lane == site: the called part sum_u c_u |s_a - u| of every CALLED
//                source individual (0 for a missing one) -- plain stores; then, only where a
//                5-8-plane ref / tgt has wide calls at the site, |s_a - v| for each wide value v
//                and every source individual, a missing one with its raw value from the table;
//   k_entry_dd   entry-driven, one thread per table entry: a missing ref / tgt call adds
//                |s_a - raw| for every source individual of its site; a missing source call adds
//                its called part sum_u c_u |raw - u| -- integer atomics, order-free and exact.
__device__ __forceinline__ int called_part(const int (&cu)[kMaxCodes], int s) {
  int d = 0;
#pragma unroll
  for (int u = 0; u < kMaxCodes; ++u) {
    const int diff = s - u;
    d += cu[u] * (diff < 0 ? -diff : diff);  // cu is 0 beyond the population's called values
  }
  return d;
}

// raw value of a missing call: entry (site, ind) of the population's table slice
__device__ __forceinline__ bool raw_lookup(const DdParams& P, const DdPop& pp, int site, int ind, int& raw) {
  int64_t lo = pp.neg_lo, hi = pp.neg_hi;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    const int s = __ldg(P.neg_site + mid);
    if (s < site || (s == site && __ldg(P.neg_ind + mid) < ind))
      lo = mid + 1;
    else
      hi = mid;
  }
  if (lo < pp.neg_hi && __ldg(P.neg_site + lo) == site && __ldg(P.neg_ind + lo) == ind) {
    raw = __ldg(P.neg_val + lo);
    return true;
  }
  return false;
}

// n (<= 8) wide values of ref (t = 0) or tgt (t = 1) at this lane's site, one byte each in `vals`,
// against every source individual.  In k_site_dd the lane owns its site's dist entries.
template <int kMaxB>
__device__ __forceinline__ void add_wide(const DdParams& P, int64_t T, int site, int lane, int t,
                                         unsigned long long vals, int n) {
  for (int k = 0; k < P.n_src; ++k) {
    const DdPop& sp = P.src[k];
    const int s_missing = (1 << sp.bits) - 1;
    const uint2* col = P.packed + ((size_t)T * P.pairs_per_site + sp.pair_off) * kTile + lane;
    for (int a0 = 0; a0 < sp.n_samples; a0 += 32) {
      uint32_t w[kMaxB];
#pragma unroll
      for (int b = 0; b < kMaxB; ++b) w[b] = b < sp.bits ? plane_word(col, (a0 >> 5) * sp.bits + b) : 0u;
      const int cnt = sp.n_samples - a0 < 32 ? sp.n_samples - a0 : 32;
      for (int bit = 0; bit < cnt; ++bit) {
        int sv = 0;
#pragma unroll
        for (int b = 0; b < kMaxB; ++b) sv |= (int)((w[b] >> bit) & 1u) << b;
        if (sv == s_missing) {
          sv = -1;
          if (!raw_lookup(P, sp, site, a0 + bit, sv)) *P.err = 1;
        }
        int d = 0;
        for (int i = 0; i < n; ++i) {
          const int diff = sv - (int)((vals >> (8 * i)) & 0xffu);
          d += diff < 0 ? -diff : diff;
        }
        P.dist[((size_t)(P.slot0[k] + a0 + bit) * 2 + t) * P.stride + site] += d;
      }
    }
  }
}

// kMaxB = 8: a min-blocks hint of 1 lets ptxas use 80 registers instead of spilling at 64
template <int kMaxB>
__global__ void __launch_bounds__(kDdWarps * 32, kMaxB > 4 ? 1 : 0) k_site_dd(const __grid_constant__ DdParams P) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int64_t T = (int64_t)blockIdx.x * kDdWarps + warp; T < P.n_tiles; T += (int64_t)gridDim.x * kDdWarps) {
    const int site = (int)(T * kTile) + lane;
    int cu[2][kMaxCodes];
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      const DdPop& pp = t == 0 ? P.ref : P.tgt;
      const int32_t* h = P.hist + (size_t)pp.code_base * P.stride + site;
      const int n_called = value_rows<kMaxB>(pp.bits);
#pragma unroll
      for (int u = 0; u < kMaxCodes; ++u) cu[t][u] = u < n_called ? __ldg(h + (size_t)u * P.stride) : 0;
    }
    for (int k = 0; k < P.n_src; ++k) {
      const DdPop& sp = P.src[k];
      const int s_missing = (1 << sp.bits) - 1;
      const uint2* col = P.packed + ((size_t)T * P.pairs_per_site + sp.pair_off) * kTile + lane;
      // called source values repeat (0, 1, 2 for two planes): their distances once per site
      int dc[2][3];
      if (sp.bits == 2) {
#pragma unroll
        for (int t = 0; t < 2; ++t)
#pragma unroll
          for (int v = 0; v < 3; ++v) dc[t][v] = called_part(cu[t], v);
      }
      for (int a0 = 0; a0 < sp.n_samples; a0 += 32) {
        uint32_t w[kMaxB];
#pragma unroll
        for (int b = 0; b < kMaxB; ++b) w[b] = b < sp.bits ? plane_word(col, (a0 >> 5) * sp.bits + b) : 0u;
        const int cnt = sp.n_samples - a0 < 32 ? sp.n_samples - a0 : 32;
        for (int bit = 0; bit < cnt; ++bit) {
          int sv = 0;
#pragma unroll
          for (int b = 0; b < kMaxB; ++b) sv |= (int)((w[b] >> bit) & 1u) << b;
          int dr = 0, dt = 0;
          if (sv != s_missing) {
            if (sp.bits == 2) {
              dr = sv == 0 ? dc[0][0] : (sv == 1 ? dc[0][1] : dc[0][2]);
              dt = sv == 0 ? dc[1][0] : (sv == 1 ? dc[1][1] : dc[1][2]);
            } else {
              dr = called_part(cu[0], sv);
              dt = called_part(cu[1], sv);
            }
          }
          int32_t* o = P.dist + (size_t)(P.slot0[k] + a0 + bit) * 2 * P.stride + site;
          o[0] = dr;
          o[P.stride] = dt;
        }
      }
    }
    if constexpr (kMaxB > 4) {
      // wide ref / tgt calls: re-read the population's planes where its wide-call row is non-zero
      for (int t = 0; t < 2; ++t) {
        const DdPop& pp = t == 0 ? P.ref : P.tgt;
        if (pp.bits <= 4) continue;
        int left = __ldg(P.hist + (size_t)(pp.code_base + kMaxCodes) * P.stride + site);
        const uint2* col = P.packed + ((size_t)T * P.pairs_per_site + pp.pair_off) * kTile + lane;
        const int G = (pp.n_samples + 31) >> 5;
        for (int g = 0; g < G && left > 0; ++g) {
          uint32_t w[kMaxB];
#pragma unroll
          for (int b = 0; b < kMaxB; ++b) w[b] = b < pp.bits ? plane_word(col, g * pp.bits + b) : 0u;
          const uint32_t low_ones = w[0] & w[1] & w[2] & w[3];
          uint32_t hi = 0, all = low_ones;
#pragma unroll
          for (int b = 4; b < kMaxB; ++b) {
            hi |= w[b];
            if (b < pp.bits) all &= w[b];
          }
          uint32_t wm = (hi | low_ones) & ~all;  // as k_site_hist's wide row
          left -= __popc(wm);
          while (wm) {
            unsigned long long vals = 0;
            int n = 0;
            for (; wm && n < 8; ++n) {
              const int bit = __ffs(wm) - 1;
              wm &= wm - 1;
              int v = 0;
#pragma unroll
              for (int b = 0; b < kMaxB; ++b) v |= (int)((w[b] >> bit) & 1u) << b;
              vals |= (unsigned long long)v << (8 * n);
            }
            add_wide<kMaxB>(P, T, site, lane, t, vals, n);
          }
        }
      }
    }
  }
}

// one thread per entry of the ref table, the tgt table and the source tables, in that order
template <int kMaxB>
__global__ void __launch_bounds__(256) k_entry_dd(const __grid_constant__ DdParams P, int64_t n_ref, int64_t n_tgt,
                                                  int64_t n_total) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_total; i += (int64_t)gridDim.x * blockDim.x) {
    if (i < n_ref + n_tgt) {
      // a missing ref / tgt call against every source individual of its site
      const int t = i < n_ref ? 0 : 1;
      const DdPop& pp = t == 0 ? P.ref : P.tgt;
      const int64_t e = pp.neg_lo + (t == 0 ? i : i - n_ref);
      const int site = __ldg(P.neg_site + e), v = __ldg(P.neg_val + e);
      if (site < 0 || site >= P.n_sites) continue;
      for (int k = 0; k < P.n_src; ++k) {
        const DdPop& sp = P.src[k];
        const int s_missing = (1 << sp.bits) - 1;
        const uint2* col = P.packed + ((size_t)(site >> 5) * P.pairs_per_site + sp.pair_off) * kTile + (site & 31);
        for (int a0 = 0; a0 < sp.n_samples; a0 += 32) {
          uint32_t w[kMaxB];
#pragma unroll
          for (int b = 0; b < kMaxB; ++b) w[b] = b < sp.bits ? plane_word(col, (a0 >> 5) * sp.bits + b) : 0u;
          const int cnt = sp.n_samples - a0 < 32 ? sp.n_samples - a0 : 32;
          for (int bit = 0; bit < cnt; ++bit) {
            int sv = 0;
#pragma unroll
            for (int b = 0; b < kMaxB; ++b) sv |= (int)((w[b] >> bit) & 1u) << b;
            if (sv == s_missing) {  // the source call is missing too: its raw value is in the table
              sv = -1;
              if (!raw_lookup(P, sp, site, a0 + bit, sv)) *P.err = 1;
            }
            const int diff = sv - v;
            atomicAdd(P.dist + ((size_t)(P.slot0[k] + a0 + bit) * 2 + t) * P.stride + site, diff < 0 ? -diff : diff);
          }
        }
      }
    } else {
      // a missing source call against the called ref / tgt values 0..14 of its site (wide ones: k_site_dd)
      int64_t r = i - n_ref - n_tgt;
      int k = 0;
      while (k + 1 < P.n_src && r >= P.src[k].neg_hi - P.src[k].neg_lo) {
        r -= P.src[k].neg_hi - P.src[k].neg_lo;
        ++k;
      }
      const int64_t e = P.src[k].neg_lo + r;
      const int site = __ldg(P.neg_site + e), a = __ldg(P.neg_ind + e), v = __ldg(P.neg_val + e);
      if (site < 0 || site >= P.n_sites || a < 0 || a >= P.src[k].n_samples) continue;
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const DdPop& pp = t == 0 ? P.ref : P.tgt;
        const int32_t* h = P.hist + (size_t)pp.code_base * P.stride + site;
        const int n_called = value_rows<kMaxB>(pp.bits);
        int d = 0;
        for (int u = 0; u < n_called; ++u) {
          const int diff = v - u;
          d += __ldg(h + (size_t)u * P.stride) * (diff < 0 ? -diff : diff);
        }
        atomicAdd(P.dist + ((size_t)(P.slot0[k] + a) * 2 + t) * P.stride + site, d);
      }
    }
  }
}

// ---- pass 3: window sums of the per-site distances ----------------------------------------------
// grid: x = windows (one warp each, grid-stride), y = source population.  Exact int64 sums.
__global__ void __launch_bounds__(kDdWarps * 32) k_window_dd(const __grid_constant__ DdParams P) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int k = blockIdx.y;
  const int m = P.src[k].n_samples;
  for (int i = blockIdx.x * kDdWarps + warp; i < P.W; i += gridDim.x * kDdWarps) {
    const int lo = (int)warp_lower_bound(P.pos, P.n_sites, P.ws[i], lane);
    int hi = (int)warp_lower_bound(P.pos, P.n_sites, P.we[i] + 1, lane);
    if (hi < lo) hi = lo;
    for (int a = 0; a < m; ++a) {
      const int32_t* dr = P.dist + (size_t)(P.slot0[k] + a) * 2 * P.stride;
      const int32_t* dt = dr + P.stride;
      long long R = 0, Tt = 0;
      int s = lo + lane;
      for (; s + 96 < hi; s += 128) {  // four coalesced loads per row in flight
        int r[4], t[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          r[u] = __ldg(dr + s + 32 * u);
          t[u] = __ldg(dt + s + 32 * u);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          R += r[u];
          Tt += t[u];
        }
      }
      for (; s < hi; s += 32) {
        R += __ldg(dr + s);
        Tt += __ldg(dt + s);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        R += __shfl_xor_sync(0xffffffffu, R, o);
        Tt += __shfl_xor_sync(0xffffffffu, Tt, o);
      }
      if (lane == 0) {
        const size_t at = ((size_t)k * P.W + i) * P.m_max + a;
        P.ref_sum[at] = R;
        P.tgt_sum[at] = Tt;
      }
    }
  }
}

// histogram rows of a population: one per called value for 2-4 planes; values 0..14 plus the
// wide-call row for 5-8 planes (a dense histogram of 255 values would take 6 GB per population
// at chromosome-1 scale)
static int32_t code_rows(const sai_pop_layout& L) { return L.bits > 4 ? kMaxCodes + 1 : (1 << L.bits) - 1; }

// a per-site distance sum_j |s - r_j| is at most 254 n (values 0..127, raw values -127..-1) and is
// kept in int32
constexpr int32_t kMaxDdSamples = 2147483647 / 254;

static bool any_wide(const sai_layout* lay, const int32_t* pops, int n) {
  for (int q = 0; q < n; ++q)
    if (lay->pop[pops[q]].bits > 4) return true;
  return false;
}

}  // namespace sai

using namespace sai;

extern "C" int64_t sai_hist_rows(const sai_layout* lay, const int32_t* pops, int32_t n) {
  if (!lay || !pops || n < 0) return 0;
  int64_t rows = 0;
  for (int q = 0; q < n; ++q) {
    if (pops[q] < 0 || pops[q] >= lay->n_pops) return 0;
    rows += code_rows(lay->pop[pops[q]]);
  }
  return rows;
}

extern "C" int sai_site_hist(const sai_layout* lay, const void* d_packed, int64_t n_sites, const int32_t* pops,
                             int32_t n_hist_pops, int32_t* d_hist, int64_t stride, uint64_t* d_missing,
                             void* stream) {
  if (int rc = validate_layout(lay)) return rc;
  SAI_REQUIRE(pops && d_hist, "NULL pointer");
  SAI_REQUIRE(n_hist_pops >= 1 && n_hist_pops <= SAI_MAX_POPS, "n_hist_pops %d outside [1,%d]", n_hist_pops,
              SAI_MAX_POPS);
  SAI_REQUIRE(n_sites >= 0 && n_sites < (1ll << 31) - 64, "n_sites out of range");
  const int64_t n_tiles = sai_num_tiles(n_sites);
  SAI_REQUIRE(stride >= n_tiles * kTile, "stride smaller than the tiled site count");
  if (n_sites == 0) return SAI_OK;
  SAI_REQUIRE(d_packed, "NULL packed matrix");
  HistParams P{};
  P.packed = static_cast<const uint2*>(d_packed);
  P.pairs_per_site = lay->pairs_per_site;
  P.n_sites = (int32_t)n_sites;
  P.n_tiles = n_tiles;
  P.stride = stride;
  P.n_slots = n_hist_pops;
  int32_t base = 0;
  for (int q = 0; q < n_hist_pops; ++q) {
    SAI_REQUIRE(pops[q] >= 0 && pops[q] < lay->n_pops, "bad population index");
    const sai_pop_layout& L = lay->pop[pops[q]];
    P.pair_off[q] = L.pair_off;
    P.n_groups[q] = L.n_groups;
    P.bits[q] = L.bits;
    P.code_base[q] = base;
    P.pad[q] = 32 * L.n_groups - L.n_samples;
    base += code_rows(L);
  }
  P.hist = d_hist;
  P.missing = reinterpret_cast<unsigned long long*>(d_missing);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (d_missing) SAI_CUDA_CHECK(cudaMemsetAsync(d_missing, 0, sizeof(uint64_t) * n_hist_pops, st));
  const int64_t want = (n_tiles + kHistWarps - 1) / kHistWarps;
  const int64_t cap = (int64_t)sm_count() * 4;  // 56 registers: 4 resident blocks per SM, one wave
  auto kernel = any_wide(lay, pops, n_hist_pops) ? k_site_hist<SAI_MAX_BITS> : k_site_hist<4>;
  kernel<<<(unsigned)(want < cap ? want : cap), kHistWarps * 32, 0, st>>>(P);
  SAI_CUDA_CHECK(cudaGetLastError());
  return SAI_OK;
}

extern "C" int sai_window_dd(const sai_layout* lay, const void* d_packed, const int32_t* d_pos, int64_t n_sites,
                             const int64_t* d_win_start, const int64_t* d_win_end, int64_t n_windows,
                             const int32_t* d_hist, int64_t stride, int32_t ref_pop, int32_t tgt_pop,
                             const int32_t* src_pops, int32_t n_src, const int64_t* neg_off,
                             const int32_t* d_neg_site, const int32_t* d_neg_ind, const int32_t* d_neg_val,
                             int64_t* d_ref_sum, int64_t* d_tgt_sum, int32_t m_max, int32_t* d_err,
                             void* stream) {
  if (int rc = validate_layout(lay)) return rc;
  SAI_REQUIRE(d_hist && d_ref_sum && d_tgt_sum && src_pops && neg_off && d_err, "NULL pointer");
  SAI_REQUIRE(n_sites >= 0 && n_sites < (1ll << 31) - 64 && stride >= n_sites, "bad n_sites / stride");
  SAI_REQUIRE(n_windows >= 0 && n_windows < (1ll << 31) - 1024, "window count out of range");
  SAI_REQUIRE(n_windows == 0 || (d_win_start && d_win_end), "NULL windows");
  SAI_REQUIRE(ref_pop >= 0 && ref_pop < lay->n_pops && tgt_pop >= 0 && tgt_pop < lay->n_pops,
              "bad population index");
  SAI_REQUIRE(n_src >= 1 && n_src <= SAI_MAX_SRC, "n_src %d outside [1,%d]", n_src, SAI_MAX_SRC);
  SAI_REQUIRE(neg_off[0] == 0, "neg_off[0] must be 0");
  for (int p = 0; p < lay->n_pops; ++p) SAI_REQUIRE(neg_off[p + 1] >= neg_off[p], "neg_off must be non-decreasing");
  SAI_REQUIRE(neg_off[lay->n_pops] == 0 || (d_neg_site && d_neg_ind && d_neg_val), "NULL negative-value table");
  SAI_REQUIRE(lay->pop[ref_pop].n_samples <= kMaxDdSamples && lay->pop[tgt_pop].n_samples <= kMaxDdSamples,
              "DD supports at most %d individuals in ref and tgt", kMaxDdSamples);
  auto fill = [&](DdPop& d, int pop, int32_t code_base) {
    const sai_pop_layout& L = lay->pop[pop];
    d.pair_off = L.pair_off;
    d.bits = L.bits;
    d.n_samples = L.n_samples;
    d.code_base = code_base;
    d.neg_lo = neg_off[pop];
    d.neg_hi = neg_off[pop + 1];
  };
  DdParams P{};
  P.packed = static_cast<const uint2*>(d_packed);
  P.pairs_per_site = lay->pairs_per_site;
  P.pos = d_pos;
  P.n_sites = (int32_t)n_sites;
  P.ws = d_win_start;
  P.we = d_win_end;
  P.W = (int32_t)n_windows;
  P.hist = d_hist;
  P.stride = stride;
  fill(P.ref, ref_pop, 0);
  fill(P.tgt, tgt_pop, code_rows(lay->pop[ref_pop]));
  P.n_src = n_src;
  for (int k = 0; k < n_src; ++k) {
    SAI_REQUIRE(src_pops[k] >= 0 && src_pops[k] < lay->n_pops, "bad source population index");
    fill(P.src[k], src_pops[k], 0);
    SAI_REQUIRE(lay->pop[src_pops[k]].n_samples <= m_max, "m_max smaller than a source population");
  }
  P.neg_site = d_neg_site;
  P.neg_ind = d_neg_ind;
  P.neg_val = d_neg_val;
  P.ref_sum = reinterpret_cast<long long*>(d_ref_sum);
  P.tgt_sum = reinterpret_cast<long long*>(d_tgt_sum);
  P.m_max = m_max;
  P.err = d_err;
  if (n_windows == 0) return SAI_OK;
  SAI_REQUIRE(n_sites == 0 || (d_packed && d_pos), "NULL input");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // per-site distances: one int32 pair (ref, tgt) per source individual and site (stream-ordered scratch)
  int32_t slots = 0;
  for (int k = 0; k < n_src; ++k) {
    P.slot0[k] = slots;
    slots += P.src[k].n_samples;
  }
  P.n_tiles = sai_num_tiles(n_sites);
  SAI_REQUIRE(stride >= P.n_tiles * kTile, "stride smaller than the tiled site count");
  void* scratch = nullptr;
  if (int rc = scratch_alloc(&scratch, sizeof(int32_t) * 2 * (size_t)slots * (size_t)std::max<int64_t>(stride, 32), st)) return rc;
  P.dist = static_cast<int32_t*>(scratch);
  if (P.n_tiles > 0) {
    const int32_t ref_tgt[2] = {ref_pop, tgt_pop};
    const bool wide = any_wide(lay, ref_tgt, 2) || any_wide(lay, src_pops, n_src);
    const int64_t wantt = (P.n_tiles + kDdWarps - 1) / kDdWarps;
    const int64_t capt = (int64_t)sm_count() * 16;
    (wide ? k_site_dd<SAI_MAX_BITS> : k_site_dd<4>)<<<(unsigned)(wantt < capt ? wantt : capt), kDdWarps * 32, 0, st>>>(P);
    SAI_CUDA_CHECK(cudaGetLastError());
    const int64_t n_ref = P.ref.neg_hi - P.ref.neg_lo, n_tgt = P.tgt.neg_hi - P.tgt.neg_lo;
    int64_t n_total = n_ref + n_tgt;
    for (int k = 0; k < n_src; ++k) n_total += P.src[k].neg_hi - P.src[k].neg_lo;
    if (n_total > 0) {
      const int64_t wante = (n_total + 255) / 256;
      const int64_t cape = (int64_t)sm_count() * 32;
      (wide ? k_entry_dd<SAI_MAX_BITS> : k_entry_dd<4>)<<<(unsigned)(wante < cape ? wante : cape), 256, 0, st>>>(P, n_ref, n_tgt, n_total);
      SAI_CUDA_CHECK(cudaGetLastError());
    }
  }
  const int64_t want = (n_windows + kDdWarps - 1) / kDdWarps;
  const int64_t cap = (int64_t)sm_count() * 16;
  const dim3 grid((unsigned)(want < cap ? want : cap), (unsigned)n_src);
  k_window_dd<<<grid, kDdWarps * 32, 0, st>>>(P);
  SAI_CUDA_CHECK(cudaGetLastError());
  return scratch_free(scratch, st);
}
