// N1: genome-wide outlier threshold of a score column (`sai outlier`, sai/sai.py:192-214) on the
// device: the linear quantile of the column's non-NaN values (pandas `Series.quantile(q)` ->
// numpy 'linear': virtual index (n-1) q, the two neighbouring order statistics, separately rounded
// lerp -- numpy/lib/_function_base_impl.py _get_indexes / _lerp).
//
// The column arrives as `n_chunks` equally long pieces (one per rank after ONE
// all_gather_into_tensor over NVLink; NaN = padding or a window without a value), so nothing is
// copied or sorted on the host.  One thread-block cluster (8 CTAs of 1024 threads, histograms
// merged through distributed shared memory) per column selects the order statistic
// exactly by an MSB-first radix select over the order-preserving 64-bit image of the doubles
// (sign-flipped, so negative statistics such as Danc / fd work too): passes with a 256-bin shared
// histogram over the L2-resident column until the selected bin fits shared memory, then the
// remaining digits there.  Everything is exact: the result equals what sorting the column gives.
#include <cooperative_groups.h>
#include <math_constants.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace sai {

constexpr int kQThreads = 1024;
constexpr int kQCluster = 8;  // CTAs (SMs) per column: one thread-block cluster, histograms merged through DSMEM

struct ColParams {
  const double* vals;
  int32_t n_chunks;
  int64_t chunk_stride;  // doubles between the pieces of one column
  int64_t col_stride;    // doubles between columns inside a piece
  int64_t len;           // doubles per piece
  double q;
  double* out;  // [n_cols][4]: threshold (NaN if undefined), n_valid, min, max
};

__device__ __forceinline__ unsigned long long ordered_key(double v) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(__dadd_rn(v, 0.0));  // -0.0 -> +0.0
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_value(unsigned long long k) {
  const unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double((long long)b);
}

// One thread-block CLUSTER of kQCluster CTAs per column (8 SMs instead of one): CTA r owns the
// elements [r*1024 + tid + j*8192]; per radix pass every CTA histograms its share in its own shared
// memory, the cluster barrier publishes the eight histograms and every CTA merges them through
// distributed shared memory, so all CTAs pick the same bin without a trip through global memory.

// f(key) for every non-NaN value of this CTA's share of the column
template <typename F>
__device__ __forceinline__ void for_each_key(const ColParams& P, int col, int rank, F f) {
  constexpr int kInFlight = 4;  // independent loads per thread
  constexpr int64_t kStride = (int64_t)kQCluster * kQThreads;
  for (int c = 0; c < P.n_chunks; ++c) {
    const double* p = P.vals + (size_t)c * P.chunk_stride + (size_t)col * P.col_stride;
    int64_t i = (int64_t)rank * kQThreads + threadIdx.x;
    for (; i + (kInFlight - 1) * kStride < P.len; i += kInFlight * kStride) {
      double v[kInFlight];
#pragma unroll
      for (int u = 0; u < kInFlight; ++u) v[u] = __ldg(p + i + u * kStride);
#pragma unroll
      for (int u = 0; u < kInFlight; ++u)
        if (v[u] == v[u]) f(ordered_key(v[u]));
    }
    for (; i < P.len; i += kStride) {
      const double v = __ldg(p + i);
      if (v == v) f(ordered_key(v));
    }
  }
}

constexpr int kQCap = 4096;  // candidate keys kept in shared memory once the selected bin is that small

struct SelectScratch {
  int hist[256];      // this CTA's histogram of the current digit (read by the whole cluster)
  int merged[256];    // the cluster's histogram
  long long bcast[4];
  unsigned long long red[kQThreads / 32];
  unsigned long long stat[3];      // this CTA's n_valid / min key / max key (read by the whole cluster)
  unsigned long long best;         // this CTA's candidate in a cluster-wide min (read by the whole cluster)
  unsigned long long keys[kQCap];  // this CTA's share of the gathered candidates
  int n_keys;
};

__device__ __forceinline__ unsigned long long block_min64(unsigned long long v, unsigned long long* s_red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned lo = __shfl_xor_sync(0xffffffffu, (unsigned)v, o);
    const unsigned hi = __shfl_xor_sync(0xffffffffu, (unsigned)(v >> 32), o);
    const unsigned long long w = ((unsigned long long)hi << 32) | lo;
    v = w < v ? w : v;
  }
  __syncthreads();
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
  __syncthreads();
  unsigned long long r = s_red[0];
  for (int w = 1; w < kQThreads / 32; ++w) r = s_red[w] < r ? s_red[w] : r;
  return r;
}

// minimum over the cluster of every CTA's block-wide minimum
__device__ __forceinline__ unsigned long long cluster_min64(cg::cluster_group& cluster, unsigned long long v, SelectScratch& S) {
  const unsigned long long mine = block_min64(v, S.red);
  if (threadIdx.x == 0) S.best = mine;
  cluster.sync();
  unsigned long long r = ~0ull;
  for (int c = 0; c < kQCluster; ++c) {
    const unsigned long long o = *cluster.map_shared_rank(&S.best, c);
    r = o < r ? o : r;
  }
  cluster.sync();  // nobody overwrites S.best while a neighbour still reads it
  return r;
}

// Exact k-th smallest key (0-based) by MSB-first radix select; count_le = number of keys <= it.
// The passes read the column from L2 until the selected bin holds <= kQCap keys; those are then
// gathered into shared memory once (every CTA keeps the candidates of its own share) and the
// remaining digits are resolved there.  n_cand = this CTA's gathered candidates (for the
// successor search): all of its keys that share the answer's prefix down to the gathering digit.
__device__ unsigned long long cluster_radix_select(cg::cluster_group& cluster, const ColParams& P, int col, int rank,
                                                   long long k, SelectScratch& S, long long& count_le, int& n_cand) {
  unsigned long long prefix = 0;
  long long kk = k, eq = 0;
  bool in_smem = false;
  int n_smem = 0;
  for (int pass = 0; pass < 8; ++pass) {
    const int shift = 56 - 8 * pass;
    if (threadIdx.x < 256) S.hist[threadIdx.x] = 0;
    __syncthreads();
    auto count = [&](unsigned long long key) {
      if (pass == 0 || (key >> (shift + 8)) == (prefix >> (shift + 8))) atomicAdd(&S.hist[(int)((key >> shift) & 255ull)], 1);
    };
    if (in_smem) {
      for (int i = threadIdx.x; i < n_smem; i += kQThreads) count(S.keys[i]);
    } else {
      for_each_key(P, col, rank, count);
    }
    cluster.sync();  // all eight histograms are complete
    // merge the eight histograms through distributed shared memory and find the bin that holds rank kk:
    // threads 0..255 own one bin each; inclusive scan = warp shuffles + the eight warp totals
    int mine = 0, incl = 0;
    if (threadIdx.x < 256) {
      for (int c = 0; c < kQCluster; ++c) mine += cluster.map_shared_rank(S.hist, c)[threadIdx.x];
      incl = mine;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, incl, o);
        if ((threadIdx.x & 31) >= o) incl += y;
      }
      if ((threadIdx.x & 31) == 31) S.merged[threadIdx.x >> 5] = incl;  // warp totals
    }
    if (threadIdx.x == 0) S.bcast[0] = 255, S.bcast[1] = 0, S.bcast[2] = 0;
    cluster.sync();  // ... the histograms are read by everybody: S.hist may be reset in the next pass
    if (threadIdx.x < 256) {
      long long before = 0;
      for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) before += S.merged[w];
      const long long hi = before + incl, lo = hi - mine;
      if (mine > 0 && kk >= lo && kk < hi) {  // exactly one bin
        S.bcast[0] = threadIdx.x;
        S.bcast[1] = lo;
        S.bcast[2] = mine;
      }
    }
    __syncthreads();
    const int bin = (int)S.bcast[0];
    const long long below = S.bcast[1], cnt = S.bcast[2];
    __syncthreads();  // S.bcast is rewritten in the next pass
    prefix |= (unsigned long long)bin << shift;
    kk -= below;
    eq = cnt;
    if (!in_smem && cnt <= kQCap && pass < 7) {  // gather the bin's keys once; finish in shared memory
      if (threadIdx.x == 0) S.n_keys = 0;
      __syncthreads();
      for_each_key(P, col, rank, [&](unsigned long long key) {
        if ((key >> shift) == (prefix >> shift)) S.keys[atomicAdd(&S.n_keys, 1)] = key;  // <= cnt <= kQCap keys in the whole cluster
      });
      __syncthreads();
      in_smem = true;
      n_smem = S.n_keys;
    }
  }
  count_le = (k - kk) + eq;
  n_cand = in_smem ? n_smem : 0;
  return prefix;
}

__global__ void __cluster_dims__(kQCluster, 1, 1) __launch_bounds__(kQThreads, 1)
    k_column_quantile(const __grid_constant__ ColParams P) {
  __shared__ SelectScratch S;
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int col = blockIdx.y;
  if (threadIdx.x == 0) {
    S.stat[0] = 0;       // n_valid
    S.stat[1] = ~0ull;   // min key
    S.stat[2] = 0;       // max key
  }
  __syncthreads();
  unsigned long long n_loc = 0, mn = ~0ull, mx = 0;
  for_each_key(P, col, rank, [&](unsigned long long key) {
    ++n_loc;
    mn = key < mn ? key : mn;
    mx = key > mx ? key : mx;
  });
  atomicAdd(&S.stat[0], n_loc);
  atomicMin(&S.stat[1], mn);
  atomicMax(&S.stat[2], mx);
  cluster.sync();
  long long n = 0;
  unsigned long long kmin = ~0ull, kmax = 0;
  for (int c = 0; c < kQCluster; ++c) {
    const unsigned long long* st = cluster.map_shared_rank(S.stat, c);
    n += (long long)st[0];
    kmin = st[1] < kmin ? st[1] : kmin;
    kmax = st[2] > kmax ? st[2] : kmax;
  }
  double thr = CUDART_NAN;
  if (n > 0 && kmin != kmax) {  // empty or single-valued column: no threshold (sai.py:195-207); cluster-uniform
    const double vi = __dmul_rn((double)(n - 1), P.q);
    long long cle;
    if (vi >= (double)(n - 1)) {
      // numpy lerps the largest value with itself: b - (b - b) (1 - g) is b for a finite b, NaN for +inf
      const double b = key_value(kmax);
      thr = __dadd_rn(b, __dsub_rn(b, b));
    } else {
      const double fl = floor(vi);
      const long long k = (long long)fl;
      const double g = __dsub_rn(vi, fl);
      int n_cand;
      const unsigned long long ka = cluster_radix_select(cluster, P, col, rank, k, S, cle, n_cand);
      unsigned long long kb = ka;
      if (k + 1 >= cle) {  // the next order statistic is the smallest key above ka
        // first among the gathered candidates: a larger key that shares ka's prefix is smaller than
        // every key outside the bin; only if ka is the bin's largest key the column is read again
        unsigned long long best = ~0ull;
        for (int i = threadIdx.x; i < n_cand; i += kQThreads) {
          const unsigned long long key = S.keys[i];
          if (key > ka && key < best) best = key;
        }
        kb = cluster_min64(cluster, best, S);
        if (kb == ~0ull) {
          best = ~0ull;
          for_each_key(P, col, rank, [&](unsigned long long key) {
            if (key > ka && key < best) best = key;
          });
          kb = cluster_min64(cluster, best, S);
        }
      }
      const double a = key_value(ka), b = key_value(kb);
      const double d = __dsub_rn(b, a);
      thr = g >= 0.5 ? __dsub_rn(b, __dmul_rn(d, __dsub_rn(1.0, g))) : __dadd_rn(a, __dmul_rn(d, g));
    }
  }
  if (rank == 0 && threadIdx.x == 0) {
    double* o = P.out + 4 * (size_t)col;
    o[0] = thr;
    o[1] = (double)n;
    o[2] = n > 0 ? key_value(kmin) : CUDART_NAN;
    o[3] = n > 0 ? key_value(kmax) : CUDART_NAN;
  }
  cluster.sync();  // no CTA leaves while a neighbour may still read its shared memory
}

}  // namespace sai

using namespace sai;

extern "C" int sai_column_quantiles(const double* d_vals, int32_t n_cols, int32_t n_chunks, int64_t chunk_stride,
                                    int64_t col_stride, int64_t len, double q, double* d_out, void* stream) {
  SAI_REQUIRE(n_cols >= 0 && n_chunks >= 1 && len >= 0 && chunk_stride >= 0 && col_stride >= 0, "bad sizes");
  SAI_REQUIRE(q >= 0.0 && q <= 1.0, "Quantiles must be in the range [0, 1]");
  if (n_cols == 0) return SAI_OK;
  SAI_REQUIRE(d_out && (len == 0 || d_vals), "NULL device pointer");
  ColParams P{d_vals, n_chunks, chunk_stride, col_stride, len, q, d_out};
  k_column_quantile<<<dim3(kQCluster, (unsigned)n_cols), kQThreads, 0, static_cast<cudaStream_t>(stream)>>>(P);
  SAI_CUDA_CHECK(cudaGetLastError());
  return SAI_OK;
}
