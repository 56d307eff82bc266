// K4: per-window U, N(Variants), exact Q and the candidate position lists (one launch).
//
// A window [start, end] (inclusive, sai/generators/window_generator.py:173-174)
// maps to the site range [lo, hi) = [lower_bound(start), lower_bound(end + 1))
// on the sorted positions; its U count is the popcount of the tile masks over
// that range (sai/stats/u_statistic.py:94-96) and Q is the numpy 'linear'
// quantile of the flagged sites' target frequencies (sai/stats/q_statistic.py:96-101;
// numpy/lib/_function_base_impl.py _lerp).  Order statistics are selected exactly
// on the float64 bit patterns (all values are non-negative, so unsigned order ==
// numeric order).
//
// One block owns a span of kSpan = 32 consecutive windows of one job.  When the
// span's starts and ends are sorted, its windows share one piece and the sites of
// all of them (R) fit the shared-memory budget, the span is scored from shared
// memory: two searches for R, a coarse index (first position of every tile of R)
// plus one 128-byte line of positions per window bound, R's masks read once with
// a prefix of their popcounts (U and the number of Q-flagged sites of a window are
// differences of it), the flagged sites of R compacted once (a window's candidates
// are a contiguous slice), a quad of threads per window for Q and the candidate
// writes, one atomic per span to reserve the candidate slices.
// Any other span -- unsorted or overlapping window lists, a span crossing pieces,
// R too long or too densely flagged -- runs the per-window code (window_batch):
// one warp per window, a cooperative 32-ary search per bound.
//
// The per-window code is issue-bound (see profiles/), so all site / tile indices
// are 32-bit (n_sites < 2^31 is checked on the host) and warp sums use REDUX.
#include <math_constants.h>
#include <stdlib.h>

#include "common.cuh"

namespace sai {

constexpr int kWinWarps = 4;
constexpr int kBufCap = 256;    // doubles buffered in shared memory per warp (more: global walk)
constexpr int kMaskCache = 64;  // tiles whose masks stay in shared memory between the two walks

struct WinParams {
  const int32_t* pos;
  int32_t n_sites;
  int32_t n_tiles;
  const int64_t* ws;
  const int64_t* we;
  const int32_t* seg_lo;  // optional: window i only sees the sites [seg_lo[i], seg_hi[i]) --
  const int32_t* seg_hi;  // several chromosomes (pieces) in one launch
  int32_t W;
  int32_t n_jobs;
  int32_t u_enabled[SAI_MAX_JOBS];
  int32_t q_enabled[SAI_MAX_JOBS];
  double quantile[SAI_MAX_JOBS];
  const uint32_t* mask_u;
  const uint32_t* mask_q;
  const double* qval;
  int64_t qval_stride;
  int32_t* nsnps;
  int64_t* u;
  double* q;
  int32_t* q_cnt;
  int64_t* u_start;  // [J][W] first candidate of the window inside the job's u_cand
  int64_t* q_start;
  unsigned long long* totals;  // [J][2] candidates reserved so far (U, Q)
  int32_t* u_cand;
  int64_t cap_u;
  int32_t* q_cand;
  int64_t cap_q;
};

__device__ __forceinline__ int clamp_key(int64_t k) {
  return k > 2147483647ll ? 2147483647 : (k < -2147483647ll ? -2147483647 : (int)k);
}

// Cooperative 32-ary lower bounds of two keys at once: first index whose
// position is >= key.  Each round probes 32 evenly spaced positions per key, so
// a 6 M-site chromosome needs 5 dependent rounds instead of 2 x 23 binary steps.
__device__ __forceinline__ void warp_lower_bound2(const int32_t* __restrict__ pos, int n,
                                                  int64_t key_a, int64_t key_b, int lane,
                                                  int& out_a, int& out_b) {
  // positions are int32: clamp the keys so that the comparisons can be 32-bit
  const int ka = clamp_key(key_a), kb = clamp_key(key_b);
  // a key beyond INT32_MAX is above every position
  int lo_a = key_a > 2147483647ll ? n : 0, hi_a = n;  // answer in [lo, hi]
  int lo_b = key_b > 2147483647ll ? n : 0, hi_b = n;
  while (hi_a > lo_a || hi_b > lo_b) {
    const int na = hi_a - lo_a, nb = hi_b - lo_b;
    const int sa = na > 32 ? (na + 31) >> 5 : 1, sb = nb > 32 ? (nb + 31) >> 5 : 1;
    const unsigned ia = (unsigned)lo_a + (unsigned)(lane + 1) * (unsigned)sa - 1u;
    const unsigned ib = (unsigned)lo_b + (unsigned)(lane + 1) * (unsigned)sb - 1u;
    const bool pa = ia < (unsigned)hi_a && __ldg(pos + ia) < ka;
    const bool pb = ib < (unsigned)hi_b && __ldg(pos + ib) < kb;
    const int ca = __popc(__ballot_sync(0xffffffffu, pa));  // sorted => the true lanes are a prefix
    const int cb = __popc(__ballot_sync(0xffffffffu, pb));
    if (na > 0) {
      // probes 0..ca-1 are < key, probe ca (if it exists) is >= key
      const unsigned nhi = (unsigned)lo_a + (unsigned)(ca + 1) * (unsigned)sa - 1u;
      lo_a += ca * sa;
      if (nhi < (unsigned)hi_a) hi_a = (int)nhi;
      if (lo_a > hi_a) lo_a = hi_a;
    }
    if (nb > 0) {
      const unsigned nhi = (unsigned)lo_b + (unsigned)(cb + 1) * (unsigned)sb - 1u;
      lo_b += cb * sb;
      if (nhi < (unsigned)hi_b) hi_b = (int)nhi;
      if (lo_b > hi_b) lo_b = hi_b;
    }
  }
  out_a = lo_a;
  out_b = lo_b;
}

__device__ __forceinline__ int warp_sum(int v) { return __reduce_add_sync(0xffffffffu, v); }
__device__ __forceinline__ int warp_excl_scan(int v, int lane) {
  int x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  return x - v;
}
__device__ __forceinline__ unsigned long long shfl64(unsigned long long v, int src) {
  unsigned lo = __shfl_sync(0xffffffffu, (unsigned)v, src);
  unsigned hi = __shfl_sync(0xffffffffu, (unsigned)(v >> 32), src);
  return ((unsigned long long)hi << 32) | lo;
}
__device__ __forceinline__ unsigned long long warp_min64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    unsigned long long w = shfl64(v, (threadIdx.x & 31) ^ o);
    v = w < v ? w : v;
  }
  return v;
}

// Site range of a window restricted to tile T: mask of the bits inside [lo, hi).
__device__ __forceinline__ uint32_t range_mask(int T, int lo, int hi) {
  const int base = T * kTile;
  uint32_t m = 0xffffffffu;
  if (lo > base) m <<= (lo - base);
  if (hi < base + kTile) m &= 0xffffffffu >> (base + kTile - hi);
  return m;
}

// Element source walking the Q mask of the window (values gathered from the
// dense qval array).  for_each calls f(key) once per flagged site, on some lane.
struct MaskSource {
  const uint32_t* mask;  // job's mask_q
  const double* qval;    // job's qval
  int lo, hi, T0, T1;
  int lane;
  template <typename F>
  __device__ __forceinline__ void for_each(F f) const {
    for (int T = T0 + lane; T <= T1; T += 32) {
      uint32_t m = __ldg(mask + T) & range_mask(T, lo, hi);
      while (m) {
        const int b = __ffs(m) - 1;
        m &= m - 1;
        f((unsigned long long)__double_as_longlong(__ldg(qval + (size_t)T * kTile + b)));
      }
    }
  }
};

struct BufSource {
  const unsigned long long* buf;
  int n;
  int lane;
  template <typename F>
  __device__ __forceinline__ void for_each(F f) const {
    for (int i = lane; i < n; i += 32) f(buf[i]);
  }
};

// Exact k-th smallest (0-based) of the source's keys by MSB-first radix select
// with a per-warp 256-bin shared histogram.  Also returns how many keys are
// <= the selected key.
template <typename Src>
__device__ unsigned long long warp_radix_select(const Src& src, int k, int* hist, int lane,
                                                int& count_le) {
  unsigned long long prefix = 0;
  int kk = k;
  int eq = 0;
  for (int pass = 0; pass < 8; ++pass) {
    const int shift = 56 - 8 * pass;
#pragma unroll
    for (int i = 0; i < 8; ++i) hist[lane * 8 + i] = 0;
    __syncwarp();
    src.for_each([&](unsigned long long key) {
      if (pass == 0 || (key >> (shift + 8)) == (prefix >> (shift + 8)))
        atomicAdd(&hist[(int)((key >> shift) & 255ull)], 1);
    });
    __syncwarp();
    int c[8], local = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      c[i] = hist[lane * 8 + i];
      local += c[i];
    }
    const int excl = warp_excl_scan(local, lane);
    const bool mine = kk >= excl && kk < excl + local;
    int bin = 0, below = 0, cnt = 0;
    if (mine) {
      int run = excl;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (cnt == 0 && kk < run + c[i]) {
          bin = lane * 8 + i;
          below = run;
          cnt = c[i];
        }
        run += c[i];
      }
    }
    const unsigned who = __ballot_sync(0xffffffffu, mine);
    const int srcl = __ffs(who) - 1;
    bin = __shfl_sync(0xffffffffu, bin, srcl);
    below = __shfl_sync(0xffffffffu, below, srcl);
    cnt = __shfl_sync(0xffffffffu, cnt, srcl);
    prefix |= (unsigned long long)bin << shift;
    kk -= below;
    eq = cnt;
    __syncwarp();
    if (cnt == 1 && pass < 7) {
      // a single key carries this prefix: fetch it and stop
      unsigned long long found = ~0ull;
      src.for_each([&](unsigned long long key) {
        if ((key >> shift) == (prefix >> shift)) found = key;
      });
      prefix = warp_min64(found);
      break;
    }
  }
  count_le = (k - kk) + eq;
  return prefix;
}

template <typename Src>
__device__ unsigned long long warp_min_above(const Src& src, unsigned long long a) {
  unsigned long long best = ~0ull;
  src.for_each([&](unsigned long long key) {
    if (key > a && key < best) best = key;
  });
  return warp_min64(best);
}

template <typename Src>
__device__ int warp_count_ge(const Src& src, double thr) {
  int c = 0;
  src.for_each([&](unsigned long long key) { c += (__longlong_as_double((long long)key) >= thr); });
  return warp_sum(c);
}

// numpy 'linear' quantile from the two neighbouring order statistics
// (_get_indexes / _get_gamma / _lerp): separately rounded, no FMA.
__device__ __forceinline__ double lerp_numpy(double a, double b, double g) {
  const double d = __dsub_rn(b, a);
  if (g >= 0.5) return __dsub_rn(b, __dmul_rn(d, __dsub_rn(1.0, g)));
  return __dadd_rn(a, __dmul_rn(d, g));
}

template <typename Src>
__device__ double warp_quantile(const Src& src, int n, double q, int* hist, int lane) {
  const double vi = __dmul_rn((double)(n - 1), q);
  int cle;
  if (vi >= (double)(n - 1)) {
    return __longlong_as_double((long long)warp_radix_select(src, n - 1, hist, lane, cle));
  }
  const double fl = floor(vi);
  const int k = (int)fl;
  const double g = __dsub_rn(vi, fl);
  const unsigned long long ka = warp_radix_select(src, k, hist, lane, cle);
  const unsigned long long kb = (k + 1 < cle) ? ka : warp_min_above(src, ka);
  return lerp_numpy(__longlong_as_double((long long)ka), __longlong_as_double((long long)kb), g);
}

// n <= 32 values, one per lane: ranks by all-pairs comparison over shuffles.
__device__ double warp_quantile_small(unsigned long long key, int n, double q, int lane) {
  int rank = 0;
  for (int j = 0; j < n; ++j) {
    const unsigned long long o = shfl64(key, j);
    rank += (o < key) || (o == key && j < lane);
  }
  const double vi = __dmul_rn((double)(n - 1), q);
  int k, k2;
  double g = 0.0;
  if (vi >= (double)(n - 1)) {
    k = k2 = n - 1;
  } else {
    const double fl = floor(vi);
    k = (int)fl;
    k2 = k + 1;
    g = __dsub_rn(vi, fl);
  }
  const unsigned ma = __ballot_sync(0xffffffffu, lane < n && rank == k);
  const unsigned mb = __ballot_sync(0xffffffffu, lane < n && rank == k2);
  const double a = __longlong_as_double((long long)shfl64(key, __ffs(ma) - 1));
  const double b = __longlong_as_double((long long)shfl64(key, __ffs(mb) - 1));
  if (k == k2) return a;
  return lerp_numpy(a, b, g);
}

// ---------------------------------------------------------------------------
// Per-warp scratch.  The batched fast path and the generic path never use it at
// the same time, so they share the bytes.
// ---------------------------------------------------------------------------
constexpr int kFastN = 32;   // flagged sites per window (U and Q each) on the fast path
constexpr int kFastTiles = 64;

template <int kBatch>
struct FastScratch {
  unsigned long long qv[kBatch][kFastN];  // flagged target frequencies (bit patterns)
  int32_t qpos[kBatch][kFastN];           // their positions
  int32_t upos[kBatch][kFastN];           // positions of the U-flagged sites
};
struct SlowScratch {
  unsigned long long buf[kBufCap];
  int hist[256];
  uint32_t mu[kMaskCache], mq[kMaskCache];
};
template <int kBatch>
union WarpScratch {
  FastScratch<kBatch> f;
  SlowScratch s;
};

struct JobView {
  const uint32_t* __restrict__ mu;
  const uint32_t* __restrict__ mq;
  const double* __restrict__ qv;
  int32_t* __restrict__ uc;
  int32_t* __restrict__ qc;
  bool want_u, want_q;
  double qq;
  int j;
};

// Generic path for one window whose site range [lo, hi) is known: any number of
// tiles and of flagged sites.
__device__ void window_generic(const WinParams& P, const JobView& J, SlowScratch& S, int i, int lo,
                               int hi, int lane) {
  const size_t item = (size_t)J.j * P.W + i;
  int u_cnt = 0, q_n = 0;
  int T0 = 0, T1 = -1;
  if (hi > lo) {
    T0 = lo >> 5;
    T1 = (hi - 1) >> 5;
    for (int Tb = T0; Tb <= T1; Tb += 32) {
      const int T = Tb + lane;
      uint32_t a = 0, b = 0;
      if (T <= T1) {
        const uint32_t rm = range_mask(T, lo, hi);
        if (J.want_u) a = __ldg(J.mu + T) & rm;
        if (J.want_q) b = __ldg(J.mq + T) & rm;
        if (T - T0 < kMaskCache) {
          S.mu[T - T0] = a;
          S.mq[T - T0] = b;
        }
      }
      u_cnt += __popc(a);
      if (__any_sync(0xffffffffu, b != 0)) {
        const int c = __popc(b);
        int w = q_n + warp_excl_scan(c, lane);
        q_n += warp_sum(c);
        while (b) {
          const int bit = __ffs(b) - 1;
          b &= b - 1;
          if (w < kBufCap)
            S.buf[w] = (unsigned long long)__double_as_longlong(__ldg(J.qv + (size_t)T * kTile + bit));
          ++w;
        }
      }
    }
    u_cnt = warp_sum(u_cnt);
    __syncwarp();
  }
  double qres = CUDART_NAN;
  int q_cand = 0;
  if (q_n > 0) {
    if (q_n <= 32) {
      const unsigned long long key = lane < q_n ? S.buf[lane] : ~0ull;
      qres = warp_quantile_small(key, q_n, J.qq, lane);
      const bool ge = lane < q_n && __longlong_as_double((long long)key) >= qres;
      q_cand = __popc(__ballot_sync(0xffffffffu, ge));
    } else if (q_n <= kBufCap) {
      BufSource src{S.buf, q_n, lane};
      qres = warp_quantile(src, q_n, J.qq, S.hist, lane);
      q_cand = warp_count_ge(src, qres);
    } else {
      MaskSource src{J.mq, J.qv, lo, hi, T0, T1, lane};
      qres = warp_quantile(src, q_n, J.qq, S.hist, lane);
      q_cand = warp_count_ge(src, qres);
    }
  }
  // reserve this window's slices of the candidate buffers (one atomic each)
  unsigned long long ub = 0, qb = 0;
  if (lane == 0) {
    if (u_cnt > 0) ub = atomicAdd(P.totals + 2 * J.j, (unsigned long long)u_cnt);
    if (q_cand > 0) qb = atomicAdd(P.totals + 2 * J.j + 1, (unsigned long long)q_cand);
    P.nsnps[item] = hi - lo;
    P.u[item] = u_cnt;
    P.q[item] = qres;
    P.q_cnt[item] = q_cand;
    P.u_start[item] = (int64_t)ub;
    P.q_start[item] = (int64_t)qb;
  }
  if (u_cnt > 0 || q_cand > 0) {
    ub = shfl64(ub, 0);
    qb = shfl64(qb, 0);
    // second walk: candidate positions in site order (u_statistic.py:95, q_statistic.py:101)
    long long uw = (long long)ub, qw = (long long)qb;
    for (int Tb = T0; Tb <= T1; Tb += 32) {
      const int T = Tb + lane;
      uint32_t a = 0, b = 0;
      if (T <= T1) {
        uint32_t m;
        if (T - T0 < kMaskCache) {
          a = S.mu[T - T0];
          m = S.mq[T - T0];
        } else {
          const uint32_t rm = range_mask(T, lo, hi);
          a = J.want_u ? (__ldg(J.mu + T) & rm) : 0u;
          m = J.want_q ? (__ldg(J.mq + T) & rm) : 0u;
        }
        while (m) {
          const int bit = __ffs(m) - 1;
          m &= m - 1;
          if (__ldg(J.qv + (size_t)T * kTile + bit) >= qres) b |= 1u << bit;
        }
      }
      if (__any_sync(0xffffffffu, a != 0)) {
        const int ca = __popc(a);
        long long wa = uw + warp_excl_scan(ca, lane);
        uw += warp_sum(ca);
        while (a) {
          const int bit = __ffs(a) - 1;
          a &= a - 1;
          if (wa < P.cap_u) J.uc[wa] = __ldg(P.pos + T * kTile + bit);
          ++wa;
        }
      }
      if (__any_sync(0xffffffffu, b != 0)) {
        const int cb = __popc(b);
        long long wb = qw + warp_excl_scan(cb, lane);
        qw += warp_sum(cb);
        while (b) {
          const int bit = __ffs(b) - 1;
          b &= b - 1;
          if (wb < P.cap_q) J.qc[wb] = __ldg(P.pos + T * kTile + bit);
          ++wb;
        }
      }
    }
  }
  __syncwarp();
}

// 32-ary lower bounds of 2*kBatch keys at once (same invariant as a single
// search: answer in [lo, hi]); every round has 2*kBatch loads in flight.
template <int kBatch>
__device__ __forceinline__ void warp_lower_bound_batch(const int32_t* __restrict__ pos,
                                                       const int (&first)[kBatch], const int (&last)[kBatch],
                                                       const int64_t (&key)[2 * kBatch], int lane,
                                                       int (&out)[2 * kBatch]) {
  int lo[2 * kBatch], hi[2 * kBatch], k32[2 * kBatch];
#pragma unroll
  for (int t = 0; t < 2 * kBatch; ++t) {
    k32[t] = clamp_key(key[t]);
    lo[t] = key[t] > 2147483647ll ? last[t >> 1] : first[t >> 1];  // search inside [first, last)
    hi[t] = last[t >> 1];
  }
  while (true) {
    bool any = false;
#pragma unroll
    for (int t = 0; t < 2 * kBatch; ++t) any = any || (hi[t] > lo[t]);
    if (!any) break;
    bool pred[2 * kBatch];
    int step[2 * kBatch];
#pragma unroll
    for (int t = 0; t < 2 * kBatch; ++t) {
      const int nn = hi[t] - lo[t];
      step[t] = nn > 32 ? (nn + 31) >> 5 : 1;
      const unsigned idx = (unsigned)lo[t] + (unsigned)(lane + 1) * (unsigned)step[t] - 1u;
      pred[t] = idx < (unsigned)hi[t] && __ldg(pos + idx) < k32[t];
    }
#pragma unroll
    for (int t = 0; t < 2 * kBatch; ++t) {
      const int c = __popc(__ballot_sync(0xffffffffu, pred[t]));
      if (hi[t] > lo[t]) {
        const unsigned nhi = (unsigned)lo[t] + (unsigned)(c + 1) * (unsigned)step[t] - 1u;
        lo[t] += c * step[t];
        if (nhi < (unsigned)hi[t]) hi[t] = (int)nhi;
        if (lo[t] > hi[t]) lo[t] = hi[t];
      }
    }
  }
#pragma unroll
  for (int t = 0; t < 2 * kBatch; ++t) out[t] = lo[t];
}

__device__ __forceinline__ JobView job_view(const WinParams& P, int j) {
  JobView J;
  J.j = j;
  J.mu = P.mask_u + (size_t)j * P.n_tiles;
  J.mq = P.mask_q + (size_t)j * P.n_tiles;
  J.qv = P.qval + (size_t)j * P.qval_stride;
  J.want_u = P.u_enabled[j] != 0;
  J.want_q = P.q_enabled[j] != 0;
  J.qq = P.quantile[j];
  J.uc = P.u_cand + (size_t)j * P.cap_u;
  J.qc = P.q_cand + (size_t)j * P.cap_q;
  return J;
}

// The per-window code: one warp, kBatch consecutive windows from i0 at once, so
// that every dependent memory round trip (window bounds, searches, masks, flagged
// values, slice reservation) is shared by kBatch windows; windows that do not fit
// the fast path (> 64 tiles or > 32 flagged sites) fall through to window_generic.
// Takes any window list: unsorted, overlapping, end < start.
template <int kBatch>
__device__ void window_batch(const WinParams& P, const JobView& J, WarpScratch<kBatch>& SC, int i0, int lane) {
  const unsigned lt_mask = (1u << lane) - 1u;
  {
    // ---- A: window bounds as keys (one coalesced load for the whole batch) ----
    int64_t key[2 * kBatch];
    {
      const int k = lane >> 1;  // lanes 0..2*kBatch-1: lane 2k -> start of window k, 2k+1 -> end+1
      int64_t mine = 0;
      if (lane < 2 * kBatch && i0 + k < P.W) mine = (lane & 1) ? P.we[i0 + k] + 1 : P.ws[i0 + k];
#pragma unroll
      for (int t = 0; t < 2 * kBatch; ++t) key[t] = (int64_t)shfl64((unsigned long long)mine, t);
    }
    // ---- B: all searches together (inside the window's own piece when pieces are given) ----
    int bnd[2 * kBatch];
    {
      int first[kBatch], last[kBatch];
#pragma unroll
      for (int k = 0; k < kBatch; ++k) {
        const bool seg = P.seg_lo != nullptr && i0 + k < P.W;
        first[k] = seg ? __ldg(P.seg_lo + i0 + k) : 0;
        last[k] = seg ? __ldg(P.seg_hi + i0 + k) : P.n_sites;
      }
      warp_lower_bound_batch<kBatch>(P.pos, first, last, key, lane, bnd);
    }
#pragma unroll
    for (int k = 0; k < kBatch; ++k)  // end < start: the reference's masks select nothing (window_generator.py:173-174)
      if (bnd[2 * k + 1] < bnd[2 * k]) bnd[2 * k + 1] = bnd[2 * k];

    // ---- C: masks of all windows ----
    uint32_t a[kBatch][2], b[kBatch][2];
    int T0[kBatch];
    bool valid[kBatch], fast[kBatch];
#pragma unroll
    for (int k = 0; k < kBatch; ++k) {
      const int lo = bnd[2 * k], hi = bnd[2 * k + 1];
      valid[k] = i0 + k < P.W;
      T0[k] = lo >> 5;
      const int T1 = hi > lo ? (hi - 1) >> 5 : T0[k] - 1;
      fast[k] = valid[k] && (T1 - T0[k] + 1 <= kFastTiles);
#pragma unroll
      for (int it = 0; it < 2; ++it) {
        const int T = T0[k] + it * 32 + lane;
        a[k][it] = b[k][it] = 0;
        if (fast[k] && T <= T1) {
          const uint32_t rm = range_mask(T, lo, hi);
          if (J.want_u) a[k][it] = __ldg(J.mu + T) & rm;
          if (J.want_q) b[k][it] = __ldg(J.mq + T) & rm;
        }
      }
    }
    int u_cnt[kBatch], q_n[kBatch];
#pragma unroll
    for (int k = 0; k < kBatch; ++k) {
      u_cnt[k] = warp_sum(__popc(a[k][0]) + __popc(a[k][1]));
      q_n[k] = warp_sum(__popc(b[k][0]) + __popc(b[k][1]));
      fast[k] = fast[k] && u_cnt[k] <= kFastN && q_n[k] <= kFastN;
    }

    // ---- D: flagged values / positions into shared memory, loads issued before any store ----
#pragma unroll
    for (int k = 0; k < kBatch; ++k) {
      if (!fast[k] || (u_cnt[k] == 0 && q_n[k] == 0)) continue;
      int wq[2], wu[2];
      {
        const int c0 = __popc(b[k][0]), c1 = __popc(b[k][1]);
        wq[0] = q_n[k] ? warp_excl_scan(c0, lane) : 0;
        wq[1] = q_n[k] ? warp_sum(c0) + warp_excl_scan(c1, lane) : 0;
        const int d0 = __popc(a[k][0]), d1 = __popc(a[k][1]);
        wu[0] = u_cnt[k] ? warp_excl_scan(d0, lane) : 0;
        wu[1] = u_cnt[k] ? warp_sum(d0) + warp_excl_scan(d1, lane) : 0;
      }
      unsigned long long vq[2] = {0ull, 0ull};
      int pq[2] = {0, 0}, pu[2] = {0, 0};
#pragma unroll
      for (int it = 0; it < 2; ++it) {
        const int site0 = (T0[k] + it * 32 + lane) * kTile;
        if (b[k][it]) {
          const int bit = __ffs(b[k][it]) - 1;
          vq[it] = (unsigned long long)__double_as_longlong(__ldg(J.qv + (size_t)site0 + bit));
          pq[it] = __ldg(P.pos + site0 + bit);
        }
        if (a[k][it]) pu[it] = __ldg(P.pos + site0 + __ffs(a[k][it]) - 1);
      }
#pragma unroll
      for (int it = 0; it < 2; ++it) {
        const int site0 = (T0[k] + it * 32 + lane) * kTile;
        if (b[k][it]) {
          SC.f.qv[k][wq[it]] = vq[it];
          SC.f.qpos[k][wq[it]] = pq[it];
          uint32_t m = b[k][it] & (b[k][it] - 1);  // further flagged sites of the same tile (rare)
          int w = wq[it] + 1;
          while (m) {
            const int bit = __ffs(m) - 1;
            m &= m - 1;
            SC.f.qv[k][w] = (unsigned long long)__double_as_longlong(__ldg(J.qv + (size_t)site0 + bit));
            SC.f.qpos[k][w] = __ldg(P.pos + site0 + bit);
            ++w;
          }
        }
        if (a[k][it]) {
          SC.f.upos[k][wu[it]] = pu[it];
          uint32_t m = a[k][it] & (a[k][it] - 1);
          int w = wu[it] + 1;
          while (m) {
            const int bit = __ffs(m) - 1;
            m &= m - 1;
            SC.f.upos[k][w] = __ldg(P.pos + site0 + bit);
            ++w;
          }
        }
      }
    }
    __syncwarp();

    // ---- E: quantiles (n <= 32: one value per lane) ----
    double qres[kBatch];
    unsigned ge[kBatch];
#pragma unroll
    for (int k = 0; k < kBatch; ++k) {
      qres[k] = CUDART_NAN;
      ge[k] = 0;
      if (fast[k] && q_n[k] > 0) {
        const unsigned long long kv = lane < q_n[k] ? SC.f.qv[k][lane] : ~0ull;
        qres[k] = warp_quantile_small(kv, q_n[k], J.qq, lane);
        ge[k] = __ballot_sync(0xffffffffu, lane < q_n[k] && __longlong_as_double((long long)kv) >= qres[k]);
      }
    }
    // ---- F: reserve the candidate slices of all fast windows with one atomic instruction ----
    unsigned long long base = 0;
    {
      int want = 0;
#pragma unroll
      for (int k = 0; k < kBatch; ++k) {
        if (lane == 2 * k && fast[k]) want = u_cnt[k];
        if (lane == 2 * k + 1 && fast[k]) want = __popc(ge[k]);
      }
      if (want > 0) base = atomicAdd(P.totals + 2 * J.j + (lane & 1), (unsigned long long)want);
    }
    // ---- G: results and candidate positions ----
#pragma unroll
    for (int k = 0; k < kBatch; ++k) {
      if (!fast[k]) continue;
      const long long ub = (long long)shfl64(base, 2 * k), qb = (long long)shfl64(base, 2 * k + 1);
      const int qc_n = __popc(ge[k]);
      if (lane == 0) {
        const size_t item = (size_t)J.j * P.W + i0 + k;
        P.nsnps[item] = bnd[2 * k + 1] - bnd[2 * k];
        P.u[item] = u_cnt[k];
        P.q[item] = qres[k];
        P.q_cnt[item] = qc_n;
        P.u_start[item] = ub;
        P.q_start[item] = qb;
      }
      if (lane < u_cnt[k] && ub + lane < P.cap_u) J.uc[ub + lane] = SC.f.upos[k][lane];
      if ((ge[k] >> lane) & 1u) {
        const long long w = qb + __popc(ge[k] & lt_mask);
        if (w < P.cap_q) J.qc[w] = SC.f.qpos[k][lane];
      }
    }
    __syncwarp();
    // ---- windows that need the generic path ----
#pragma unroll
    for (int k = 0; k < kBatch; ++k) {
      if (valid[k] && !fast[k]) window_generic(P, J, SC.s, i0 + k, bnd[2 * k], bnd[2 * k + 1], lane);
    }
  }
}

// grid: x = window batches (kWinWarps * kBatch windows per block, grid-stride), y = job.
// Every window through window_batch: the -DSAI_EXPERIMENTS variants.
template <int kBatch, int kMinBlocks>
__global__ void __launch_bounds__(kWinWarps * 32, kMinBlocks)
    k_window_stats(const __grid_constant__ WinParams P) {
  __shared__ WarpScratch<kBatch> s_scratch[kWinWarps];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const JobView J = job_view(P, blockIdx.y);
  for (int i0 = (blockIdx.x * kWinWarps + warp) * kBatch; i0 < P.W; i0 += gridDim.x * kWinWarps * kBatch)
    window_batch<kBatch>(P, J, s_scratch[warp], i0, lane);
}

// ---------------------------------------------------------------------------
// Span path: one block per span of kSpan consecutive windows of one job.
// ---------------------------------------------------------------------------
constexpr int kSpan = 32;          // windows per span: one per lane of warp 0
constexpr int kSpanWarps = 4;
constexpr int kSpanThreads = kSpanWarps * 32;
constexpr int kSpanTiles = 512;    // tiles of the span's site range R held in shared memory
constexpr int kSpanFlags = 1024;   // U-flagged and Q-flagged sites of R held in shared memory (each)
constexpr int kSpanBlocksPerSM = 6;  // ~33 KB of shared memory per block
constexpr int kTilesPerThread = kSpanTiles / kSpanThreads;
constexpr int kKeysPerWarp = 2 * kSpan / kSpanWarps;
static_assert(kSpan == 32 && kSpanThreads == 4 * kSpan && kSpanTiles % kSpanThreads == 0 && (2 * kSpan) % kSpanWarps == 0, "span shape");

struct SpanCtl {  // outside the union: read by every warp after the fallback warps start writing their scratch
  int ok, lo, hi, T0, nT, nu, nq;
  int warp_u[kSpanWarps], warp_q[kSpanWarps];
};
struct SpanData {
  int32_t first_pos[kSpanTiles];         // coarse index: position of the first site of R in every tile
  uint32_t mu[kSpanTiles + 1], mq[kSpanTiles + 1];  // masks restricted to R (+ a zero past the end)
  int32_t pu[kSpanTiles + 1], pq[kSpanTiles + 1];   // exclusive prefix of their popcounts
  int32_t upos[kSpanFlags];              // U-flagged sites of R in site order (index, then position)
  int32_t qpos[kSpanFlags];              // Q-flagged sites of R (index, then position)
  unsigned long long qv[kSpanFlags];     // ... and their target frequencies (bit patterns)
  int64_t key[2 * kSpan];                // window k: key 2k = start, 2k + 1 = end + 1
  int32_t tile_of_key[2 * kSpan];
  int32_t bnd[2 * kSpan];
  int32_t u_a[kSpan], q_a[kSpan], n_u[kSpan], n_q[kSpan], q_c[kSpan], nsnps[kSpan];
  double qres[kSpan];
  long long u_st[kSpan], q_st[kSpan];
  int hist[kSpanWarps][256];
};
union SpanSmem {
  SpanData d;
  WarpScratch<1> w[kSpanWarps];  // the per-window fallback
};

// flagged sites of R before site x (x in [lo, hi] of R): prefix of the tile + bits below x in its tile
__device__ __forceinline__ int flags_before(const uint32_t* m, const int32_t* pre, int x, int T0) {
  const int t = (x >> 5) - T0;
  return pre[t] + __popc(m[t] & ((1u << (x & 31)) - 1u));
}

// grid: x = spans (grid-stride), y = job.  A span qualifies when its starts and its ends + 1 are
// non-decreasing, all its windows share one piece, R (the sites of all its windows) spans at most
// kSpanTiles tiles and holds at most kSpanFlags U- and Q-flagged sites.  Then every window's site
// bounds, U, Q and candidates come out of shared memory with a fixed number of dependent memory trips
// per span; any other span runs window_batch<1> per window, warp by warp.
__global__ void __launch_bounds__(kSpanThreads, kSpanBlocksPerSM) k_window_spans(const __grid_constant__ WinParams P) {
  __shared__ SpanSmem sm;
  __shared__ SpanCtl ctl;
  SpanData& S = sm.d;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const JobView J = job_view(P, blockIdx.y);
  const int n_spans = (P.W + kSpan - 1) / kSpan;

  for (int span = blockIdx.x; span < n_spans; span += gridDim.x) {
    const int i0 = span * kSpan;
    const int nw = min(kSpan, P.W - i0);
    __syncthreads();  // the previous span is done with the shared memory
    // ---- 1: qualify the span and find its site range R = [lo, hi) with two searches ----
    if (warp == 0) {
      const bool v = lane < nw;
      const int64_t ks = v ? P.ws[i0 + lane] : 0, ke = v ? P.we[i0 + lane] + 1 : 0;
      const int sl = (P.seg_lo != nullptr && v) ? P.seg_lo[i0 + lane] : 0;
      const int sh = (P.seg_lo != nullptr && v) ? P.seg_hi[i0 + lane] : P.n_sites;
      const int64_t ps = (int64_t)shfl64((unsigned long long)ks, lane - 1 < 0 ? 0 : lane - 1);
      const int64_t pe = (int64_t)shfl64((unsigned long long)ke, lane - 1 < 0 ? 0 : lane - 1);
      const int psl = __shfl_sync(0xffffffffu, sl, lane - 1 < 0 ? 0 : lane - 1);
      const int psh = __shfl_sync(0xffffffffu, sh, lane - 1 < 0 ? 0 : lane - 1);
      bool ok = !__any_sync(0xffffffffu, v && lane > 0 && (ks < ps || ke < pe || sl != psl || sh != psh));
      S.key[2 * lane] = ks;
      S.key[2 * lane + 1] = ke;
      // every key of the span lies in [min(start, end + 1) of the first window, max(...) of the last]
      const int64_t kmin = (int64_t)shfl64((unsigned long long)(ks < ke ? ks : ke), 0);
      const int64_t kmax = (int64_t)shfl64((unsigned long long)(ks > ke ? ks : ke), nw - 1);
      int lo = 0, hi = 0, T0 = 0, nT = 0;
      if (ok) {
        const int first[1] = {__shfl_sync(0xffffffffu, sl, 0)}, last[1] = {__shfl_sync(0xffffffffu, sh, 0)};
        const int64_t key[2] = {kmin, kmax};
        int out[2];
        warp_lower_bound_batch<1>(P.pos, first, last, key, lane, out);
        lo = out[0];
        hi = out[1] > lo ? out[1] : lo;
        T0 = lo >> 5;
        nT = hi > lo ? ((hi - 1) >> 5) - T0 + 1 : 0;
        ok = nT <= kSpanTiles;
      }
      if (lane == 0) {
        ctl.ok = ok;
        ctl.lo = lo;
        ctl.hi = hi;
        ctl.T0 = T0;
        ctl.nT = nT;
      }
    }
    __syncthreads();
    if (!ctl.ok) {
      for (int k = warp; k < nw; k += kSpanWarps) window_batch<1>(P, J, sm.w[warp], i0 + k, lane);
      continue;
    }
    const int lo = ctl.lo, hi = ctl.hi, T0 = ctl.T0, nT = ctl.nT;

    // ---- 2: masks of R's tiles and the coarse index, once; block-wide prefix of the popcounts ----
    {
      uint32_t a[kTilesPerThread], b[kTilesPerThread];
      int fp[kTilesPerThread];
      int su = 0, sq = 0;
#pragma unroll
      for (int r = 0; r < kTilesPerThread; ++r) {
        const int t = tid * kTilesPerThread + r, T = T0 + t;
        a[r] = b[r] = 0;
        fp[r] = 0;
        if (t < nT) {
          const uint32_t rm = range_mask(T, lo, hi);
          if (J.want_u) a[r] = __ldg(J.mu + T) & rm;
          if (J.want_q) b[r] = __ldg(J.mq + T) & rm;
          fp[r] = __ldg(P.pos + (T * kTile > lo ? T * kTile : lo));
        }
        su += __popc(a[r]);
        sq += __popc(b[r]);
      }
      const int xu = warp_excl_scan(su, lane), xq = warp_excl_scan(sq, lane);
      if (lane == 31) {
        ctl.warp_u[warp] = xu + su;
        ctl.warp_q[warp] = xq + sq;
      }
      __syncthreads();
      int bu = xu, bq = xq;
      for (int w = 0; w < warp; ++w) {
        bu += ctl.warp_u[w];
        bq += ctl.warp_q[w];
      }
#pragma unroll
      for (int r = 0; r < kTilesPerThread; ++r) {
        const int t = tid * kTilesPerThread + r;
        S.mu[t] = a[r];
        S.mq[t] = b[r];
        S.pu[t] = bu;
        S.pq[t] = bq;
        S.first_pos[t] = fp[r];
        bu += __popc(a[r]);
        bq += __popc(b[r]);
      }
      if (tid == kSpanThreads - 1) {
        S.mu[kSpanTiles] = S.mq[kSpanTiles] = 0;
        S.pu[kSpanTiles] = bu;
        S.pq[kSpanTiles] = bq;
        ctl.nu = bu;
        ctl.nq = bq;
      }
    }
    __syncthreads();
    if (ctl.nu > kSpanFlags || ctl.nq > kSpanFlags) {
      for (int k = warp; k < nw; k += kSpanWarps) window_batch<1>(P, J, sm.w[warp], i0 + k, lane);
      continue;
    }
    const int nu = ctl.nu, nq = ctl.nq;

    // ---- 3: flagged sites of R in site order; each key's tile from the coarse index ----
#pragma unroll
    for (int r = 0; r < kTilesPerThread; ++r) {
      const int t = tid * kTilesPerThread + r, site0 = (T0 + t) * kTile;
      uint32_t m = S.mu[t];
      for (int w = S.pu[t]; m; ++w, m &= m - 1) S.upos[w] = site0 + __ffs(m) - 1;
      m = S.mq[t];
      for (int w = S.pq[t]; m; ++w, m &= m - 1) S.qpos[w] = site0 + __ffs(m) - 1;
    }
    if (tid < 2 * nw) {
      // number of tiles whose first site of R lies below the key; the key's bound is inside the last of them
      const int k32 = clamp_key(S.key[tid]);
      int a = 0, b = nT;
      while (a < b) {
        const int m = (a + b) >> 1;
        if (S.first_pos[m] < k32) a = m + 1; else b = m;
      }
      S.tile_of_key[tid] = a;
    }
    __syncthreads();

    // ---- 4: flagged positions / values and every window bound: every load issued before any is used ----
    {
      int kp[kKeysPerWarp];  // the key's tile line of positions (INT32_MAX outside R: never below a key)
#pragma unroll
      for (int r = 0; r < kKeysPerWarp; ++r) {
        const int kk = warp * kKeysPerWarp + r;
        const int c = kk < 2 * nw ? S.tile_of_key[kk] : 0;
        const int idx = (T0 + c - 1) * kTile + lane;
        kp[r] = c > 0 && idx >= lo && idx < hi ? __ldg(P.pos + idx) : 2147483647;
      }
      int pu = 0, pq = 0;
      unsigned long long vq = 0;
      if (tid < nu) pu = __ldg(P.pos + S.upos[tid]);
      if (tid < nq) {
        const int site = S.qpos[tid];
        vq = (unsigned long long)__double_as_longlong(__ldg(J.qv + (size_t)site));
        pq = __ldg(P.pos + site);
      }
#pragma unroll
      for (int r = 0; r < kKeysPerWarp; ++r) {
        const int kk = warp * kKeysPerWarp + r;
        const int c = __popc(__ballot_sync(0xffffffffu, kk < 2 * nw && kp[r] < clamp_key(S.key[kk])));
        if (lane == 0 && kk < 2 * nw) {
          const int tc = S.tile_of_key[kk];
          const int base = tc > 0 ? max((T0 + tc - 1) * kTile, lo) : lo;
          // a key beyond INT32_MAX lies above every position: the end of the piece, which is hi
          S.bnd[kk] = S.key[kk] > 2147483647ll ? hi : base + c;
        }
      }
      if (tid < nu) S.upos[tid] = pu;
      if (tid < nq) {
        S.qv[tid] = vq;
        S.qpos[tid] = pq;
      }
    }
    for (int i = tid + kSpanThreads; i < nu; i += kSpanThreads) S.upos[i] = __ldg(P.pos + S.upos[i]);
    for (int i = tid + kSpanThreads; i < nq; i += kSpanThreads) {
      const int site = S.qpos[i];
      S.qv[i] = (unsigned long long)__double_as_longlong(__ldg(J.qv + (size_t)site));
      S.qpos[i] = __ldg(P.pos + site);
    }
    __syncthreads();

    // ---- 5: U, N(Variants) and Q of every window: a quad of threads per window, all windows at once ----
    {
      const int k = tid >> 2, q = tid & 3;
      const bool v = k < nw;
      int wlo = 0, whi = 0, ua = 0, ub = 0, qa = 0, qn = 0;
      if (v) {
        wlo = S.bnd[2 * k];
        whi = max(S.bnd[2 * k + 1], wlo);  // end < start selects nothing
        ua = flags_before(S.mu, S.pu, wlo, T0);
        ub = flags_before(S.mu, S.pu, whi, T0);
        qa = flags_before(S.mq, S.pq, wlo, T0);
        qn = flags_before(S.mq, S.pq, whi, T0) - qa;
      }
      // n <= 32: the two neighbouring order statistics by rank (ties broken by site order, as in
      // warp_quantile_small), the ranks of the window's values split over the quad
      const bool small = v && qn > 0 && qn <= 32;
      int ka = 0, kb = 0;
      double g = 0.0;
      if (small) {
        const double vi = __dmul_rn((double)(qn - 1), J.qq);
        if (vi >= (double)(qn - 1)) {
          ka = kb = qn - 1;
        } else {
          const double fl = floor(vi);
          ka = (int)fl;
          kb = ka + 1;
          g = __dsub_rn(vi, fl);
        }
      }
      unsigned long long va = 0, vb = 0;
      if (small) {
        for (int i = q; i < qn; i += 4) {
          const unsigned long long key = S.qv[qa + i];
          int r = 0;
          for (int j = 0; j < qn; ++j) {
            const unsigned long long o = S.qv[qa + j];
            r += (o < key) || (o == key && j < i);
          }
          if (r == ka) va = key;
          if (r == kb) vb = key;
        }
      }
      // each rank belongs to exactly one value: OR over the quad collects it
      va |= shfl64(va, lane ^ 1);
      va |= shfl64(va, lane ^ 2);
      vb |= shfl64(vb, lane ^ 1);
      vb |= shfl64(vb, lane ^ 2);
      double qres = CUDART_NAN;
      int qc = 0;
      if (small) {
        const double da = __longlong_as_double((long long)va), db = __longlong_as_double((long long)vb);
        qres = ka == kb ? da : lerp_numpy(da, db, g);
        for (int i = q; i < qn; i += 4) qc += __longlong_as_double((long long)S.qv[qa + i]) >= qres;
      }
      qc += __shfl_xor_sync(0xffffffffu, qc, 1);
      qc += __shfl_xor_sync(0xffffffffu, qc, 2);
      if (v && q == 0) {
        S.nsnps[k] = whi - wlo;
        S.u_a[k] = ua;
        S.n_u[k] = ub - ua;
        S.q_a[k] = qa;
        S.n_q[k] = qn;
        S.q_c[k] = qc;
        S.qres[k] = qres;
      }
    }
    __syncthreads();
    // windows above 32 Q-flagged sites: exact radix selection on the window's slice, warp per window
    for (int k = warp; k < nw; k += kSpanWarps) {
      const int qn = S.n_q[k];
      if (qn <= 32) continue;
      BufSource src{S.qv + S.q_a[k], qn, lane};
      const double qres = warp_quantile(src, qn, J.qq, S.hist[warp], lane);
      const int qc = warp_count_ge(src, qres);
      if (lane == 0) {
        S.qres[k] = qres;
        S.q_c[k] = qc;
      }
    }
    __syncthreads();

    // ---- 6: one atomic per span and array, coalesced result stores ----
    if (warp == 0) {
      const bool v = lane < nw;
      const int nu_k = v ? S.n_u[lane] : 0, qc_k = v ? S.q_c[lane] : 0;
      const int xu = warp_excl_scan(nu_k, lane), xq = warp_excl_scan(qc_k, lane);
      const int tu = warp_sum(nu_k), tq = warp_sum(qc_k);
      unsigned long long base = 0;
      if (lane < 2 && (lane ? tq : tu) > 0) base = atomicAdd(P.totals + 2 * J.j + lane, (unsigned long long)(lane ? tq : tu));
      const long long ubase = (long long)shfl64(base, 0), qbase = (long long)shfl64(base, 1);
      if (v) {
        const size_t item = (size_t)J.j * P.W + i0 + lane;
        const long long us = nu_k > 0 ? ubase + xu : 0, qs = qc_k > 0 ? qbase + xq : 0;
        P.nsnps[item] = S.nsnps[lane];
        P.u[item] = nu_k;
        P.q[item] = S.qres[lane];
        P.q_cnt[item] = qc_k;
        P.u_start[item] = us;
        P.q_start[item] = qs;
        S.u_st[lane] = us;
        S.q_st[lane] = qs;
      }
    }
    __syncthreads();

    // ---- 7: candidate positions in site order, a quad of threads per window ----
    {
      const int k = tid >> 2, q = tid & 3;
      int ua = 0, un = 0, qa = 0, qn = 0;
      long long us = 0, qw = 0;
      double qres = 0.0;
      if (k < nw) {
        ua = S.u_a[k];
        un = S.n_u[k];
        us = S.u_st[k];
        qa = S.q_a[k];
        qn = S.n_q[k];
        qw = S.q_st[k];
        qres = S.qres[k];
      }
      for (int e = q; e < un; e += 4)
        if (us + e < P.cap_u) J.uc[us + e] = S.upos[ua + e];
      const int steps = (int)__reduce_max_sync(0xffffffffu, (unsigned)(qn + 3) >> 2);
      for (int st = 0; st < steps; ++st) {
        const int e = 4 * st + q;
        const bool ge = e < qn && __longlong_as_double((long long)S.qv[qa + e]) >= qres;
        const unsigned m = (__ballot_sync(0xffffffffu, ge) >> (lane & 28)) & 0xfu;  // this quad's 4 bits
        const long long w = qw + __popc(m & ((1u << q) - 1u));
        if (ge && w < P.cap_q) J.qc[w] = S.qpos[qa + e];
        qw += __popc(m);
      }
    }
  }
}

}  // namespace sai

using namespace sai;

static int window_stats_impl(const int32_t* d_pos, int64_t n_sites, const int64_t* d_win_start,
                             const int64_t* d_win_end, const int32_t* d_seg_lo, const int32_t* d_seg_hi,
                             int64_t n_windows, const sai_job* jobs,
                             int32_t n_jobs, const uint32_t* d_mask_u, const uint32_t* d_mask_q,
                             const double* d_qval, int64_t qval_stride, int32_t* d_nsnps,
                             int64_t* d_u, double* d_q, int32_t* d_q_cnt, int64_t* d_u_start,
                             int64_t* d_q_start, int64_t* d_totals, int32_t* d_u_cand,
                             int64_t cap_u, int32_t* d_q_cand, int64_t cap_q, void* stream) {
  SAI_REQUIRE(d_pos && d_mask_u && d_mask_q && d_qval && d_totals, "NULL device pointer");
  SAI_REQUIRE(n_sites >= 0 && n_sites < (1ll << 31) - 64, "n_sites out of range");
  SAI_REQUIRE(n_windows >= 0 && n_windows < (1ll << 31) - 1024, "window count out of range");
  SAI_REQUIRE(jobs && n_jobs >= 1 && n_jobs <= SAI_MAX_JOBS, "n_jobs %d outside [1,%d]", n_jobs,
              SAI_MAX_JOBS);
  SAI_REQUIRE(qval_stride >= n_sites, "qval_stride too small");
  SAI_REQUIRE(n_windows == 0 || (d_win_start && d_win_end && d_nsnps && d_u && d_q && d_q_cnt &&
                                 d_u_start && d_q_start),
              "NULL device pointer");
  SAI_REQUIRE(cap_u >= 0 && cap_q >= 0 && (cap_u == 0 || d_u_cand) && (cap_q == 0 || d_q_cand),
              "bad candidate buffers");
  WinParams P{};
  P.pos = d_pos;
  P.n_sites = (int32_t)n_sites;
  P.n_tiles = (int32_t)sai_num_tiles(n_sites);
  P.ws = d_win_start;
  P.we = d_win_end;
  P.seg_lo = d_seg_lo;
  P.seg_hi = d_seg_hi;
  P.W = (int32_t)n_windows;
  P.n_jobs = n_jobs;
  for (int j = 0; j < n_jobs; ++j) {
    P.u_enabled[j] = jobs[j].u.enabled;
    P.q_enabled[j] = jobs[j].q.enabled;
    P.quantile[j] = jobs[j].quantile;
    if (jobs[j].q.enabled)
      SAI_REQUIRE(jobs[j].quantile >= 0.0 && jobs[j].quantile <= 1.0,
                  "Quantiles must be in the range [0, 1]");
  }
  P.mask_u = d_mask_u;
  P.mask_q = d_mask_q;
  P.qval = d_qval;
  P.qval_stride = qval_stride;
  P.nsnps = d_nsnps;
  P.u = d_u;
  P.q = d_q;
  P.q_cnt = d_q_cnt;
  P.u_start = d_u_start;
  P.q_start = d_q_start;
  P.totals = reinterpret_cast<unsigned long long*>(d_totals);
  P.u_cand = d_u_cand;
  P.cap_u = cap_u;
  P.q_cand = d_q_cand;
  P.cap_q = cap_q;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SAI_CUDA_CHECK(cudaMemsetAsync(d_totals, 0, sizeof(int64_t) * 2 * n_jobs, st));
  if (n_windows == 0) return SAI_OK;
#ifdef SAI_EXPERIMENTS
  // tuning knobs of tools/ builds: every window on the per-window path, windows per warp and the
  // occupancy bound
  const int64_t cap = (int64_t)sm_count() * 32;
  static const int batch = [] {
    const char* e = getenv("SAI_WIN_BATCH");
    const int b = e ? atoi(e) : 1;
    return (b == 2 || b == 4) ? b : 1;
  }();
  static const int minb = [] {
    const char* e = getenv("SAI_WIN_MINB");
    return e ? atoi(e) : 12;
  }();
  const int64_t per_block = kWinWarps * batch;
  const int64_t want = (n_windows + per_block - 1) / per_block;
  const dim3 grid((unsigned)(want < cap ? want : cap), (unsigned)n_jobs);
  if (batch == 1 && minb == 10)
    k_window_stats<1, 10><<<grid, kWinWarps * 32, 0, st>>>(P);
  else if (batch == 1 && minb == 12)
    k_window_stats<1, 12><<<grid, kWinWarps * 32, 0, st>>>(P);
  else if (batch == 1)
    k_window_stats<1, 8><<<grid, kWinWarps * 32, 0, st>>>(P);
  else if (batch == 2)
    k_window_stats<2, 6><<<grid, kWinWarps * 32, 0, st>>>(P);
  else
    k_window_stats<4, 4><<<grid, kWinWarps * 32, 0, st>>>(P);
#else
  // one block per span of kSpan windows, as many blocks as are resident at once (grid-stride)
  const int64_t spans = (n_windows + kSpan - 1) / kSpan, span_cap = (int64_t)sm_count() * kSpanBlocksPerSM;
  const dim3 grid((unsigned)(spans < span_cap ? spans : span_cap), (unsigned)n_jobs);
  // kSpanBlocksPerSM blocks of ~33 KB need the largest shared-memory carveout
  static const cudaError_t carveout = cudaFuncSetAttribute(
      k_window_spans, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  SAI_CUDA_CHECK(carveout);
  k_window_spans<<<grid, kSpanThreads, 0, st>>>(P);
#endif
  SAI_CUDA_CHECK(cudaGetLastError());
  return SAI_OK;
}

extern "C" int sai_window_stats(const int32_t* d_pos, int64_t n_sites, const int64_t* d_win_start,
                                const int64_t* d_win_end, int64_t n_windows, const sai_job* jobs,
                                int32_t n_jobs, const uint32_t* d_mask_u, const uint32_t* d_mask_q,
                                const double* d_qval, int64_t qval_stride, int32_t* d_nsnps,
                                int64_t* d_u, double* d_q, int32_t* d_q_cnt, int64_t* d_u_start,
                                int64_t* d_q_start, int64_t* d_totals, int32_t* d_u_cand,
                                int64_t cap_u, int32_t* d_q_cand, int64_t cap_q, void* stream) {
  return window_stats_impl(d_pos, n_sites, d_win_start, d_win_end, nullptr, nullptr, n_windows, jobs, n_jobs,
                           d_mask_u, d_mask_q, d_qval, qval_stride, d_nsnps, d_u, d_q, d_q_cnt, d_u_start,
                           d_q_start, d_totals, d_u_cand, cap_u, d_q_cand, cap_q, stream);
}

extern "C" int sai_window_stats_pieces(const int32_t* d_pos, int64_t n_sites, const int64_t* d_win_start,
                                       const int64_t* d_win_end, const int32_t* d_win_first_site,
                                       const int32_t* d_win_last_site, int64_t n_windows, const sai_job* jobs,
                                       int32_t n_jobs, const uint32_t* d_mask_u, const uint32_t* d_mask_q,
                                       const double* d_qval, int64_t qval_stride, int32_t* d_nsnps,
                                       int64_t* d_u, double* d_q, int32_t* d_q_cnt, int64_t* d_u_start,
                                       int64_t* d_q_start, int64_t* d_totals, int32_t* d_u_cand,
                                       int64_t cap_u, int32_t* d_q_cand, int64_t cap_q, void* stream) {
  SAI_REQUIRE(n_windows == 0 || (d_win_first_site && d_win_last_site), "NULL piece bounds");
  return window_stats_impl(d_pos, n_sites, d_win_start, d_win_end, d_win_first_site, d_win_last_site, n_windows,
                           jobs, n_jobs, d_mask_u, d_mask_q, d_qval, qval_stride, d_nsnps, d_u, d_q, d_q_cnt,
                           d_u_start, d_q_start, d_totals, d_u_cand, cap_u, d_q_cand, cap_q, stream);
}
