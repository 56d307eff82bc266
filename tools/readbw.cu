// Read-bandwidth ceiling probe (not part of the product): how fast can ANY kernel stream the
// packed matrix out of HBM on this GPU?  Gives k_site's roofline a second, read-only denominator
// next to the driver-measured copy bandwidth.
//   mode 0: flat grid-stride, 16 B per thread per load, 4 loads in flight
//   mode 1: k_site's access pattern (one warp per 20 KB tile, 8 B per lane, 8 loads in flight), XOR only
//   mode 2: like 1 with 16 loads in flight
//   mode 6: a scan of the sources alone: the last pair of every tile (the bench layout's source), 8 tiles in flight
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

__device__ __forceinline__ uint2 ld_stream(const uint2* p) {
  uint2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
  return r;
}
__device__ __forceinline__ uint4 ld_stream16(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}

__global__ void __launch_bounds__(256) k_flat(const uint4* __restrict__ p, size_t n, uint32_t* out) {
  uint32_t acc = 0;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < n; i += 4 * stride) {
    uint4 a = ld_stream16(p + i), b = ld_stream16(p + i + stride), c = ld_stream16(p + i + 2 * stride), d = ld_stream16(p + i + 3 * stride);
    acc ^= a.x ^ a.y ^ a.z ^ a.w ^ b.x ^ b.y ^ b.z ^ b.w ^ c.x ^ c.y ^ c.z ^ c.w ^ d.x ^ d.y ^ d.z ^ d.w;
  }
  for (; i < n; i += stride) {
    uint4 a = ld_stream16(p + i);
    acc ^= a.x ^ a.y ^ a.z ^ a.w;
  }
  if (acc == 0x12345678u) out[0] = acc;
}

template <int INFLIGHT>
__global__ void __launch_bounds__(256) k_tiles(const uint2* __restrict__ p, int64_t n_tiles, int pps, uint32_t* out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t acc = 0;
  for (int64_t t = (int64_t)blockIdx.x * 8 + warp; t < n_tiles; t += (int64_t)gridDim.x * 8) {
    const uint2* col = p + (size_t)t * pps * 32 + lane;
    int q = 0;
    for (; q + INFLIGHT <= pps; q += INFLIGHT) {
      uint2 v[INFLIGHT];
#pragma unroll
      for (int i = 0; i < INFLIGHT; ++i) v[i] = ld_stream(col + (size_t)(q + i) * 32);
#pragma unroll
      for (int i = 0; i < INFLIGHT; ++i) acc ^= v[i].x ^ v[i].y;
    }
    for (; q < pps; ++q) {
      uint2 v = ld_stream(col + (size_t)q * 32);
      acc ^= v.x ^ v.y;
    }
  }
  if (acc == 0x12345678u) out[0] = acc;
}

__device__ __forceinline__ uint32_t xor3(uint32_t a, uint32_t b, uint32_t c) { uint32_t r; asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
__device__ __forceinline__ uint32_t maj3(uint32_t a, uint32_t b, uint32_t c) { uint32_t r; asm("lop3.b32 %0, %1, %2, %3, 0xE8;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
struct SliceCounter {
  uint32_t ones = 0, twos = 0, fours = 0; int high = 0;
  __device__ __forceinline__ void add8(const uint32_t (&w)[8]) {
    uint32_t tA = maj3(ones, w[0], w[1]); ones = xor3(ones, w[0], w[1]);
    uint32_t tB = maj3(ones, w[2], w[3]); ones = xor3(ones, w[2], w[3]);
    uint32_t fA = maj3(twos, tA, tB); twos = xor3(twos, tA, tB);
    tA = maj3(ones, w[4], w[5]); ones = xor3(ones, w[4], w[5]);
    tB = maj3(ones, w[6], w[7]); ones = xor3(ones, w[6], w[7]);
    uint32_t fB = maj3(twos, tA, tB); twos = xor3(twos, tA, tB);
    uint32_t e = maj3(fours, fA, fB); fours = xor3(fours, fA, fB);
    high += __popc(e);
  }
  __device__ __forceinline__ int total() const { return 8 * high + 4 * __popc(fours) + 2 * __popc(twos) + __popc(ones); }
};
// mode 3 / 4: k_site's loads + its carry-save adders (3 streams / 2 streams + OR of a&b), nothing else
template <bool SKIPM>
__global__ void __launch_bounds__(256) k_csa(const uint2* __restrict__ p, int64_t n_tiles, int pps, uint32_t* out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t acc = 0;
  for (int64_t t = (int64_t)blockIdx.x * 8 + warp; t < n_tiles; t += (int64_t)gridDim.x * 8) {
    const uint2* col = p + (size_t)t * pps * 32 + lane;
    SliceCounter ca, cb, cm;
    for (int q = 0; q + 8 <= pps; q += 8) {
      uint2 v[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = ld_stream(col + (size_t)(q + i) * 32);
      uint32_t a[8], b[8], m[8], mo = 0;
#pragma unroll
      for (int i = 0; i < 8; ++i) { a[i] = v[i].x; b[i] = v[i].y; m[i] = v[i].x & v[i].y; mo |= m[i]; }
      ca.add8(a); cb.add8(b);
      if (!SKIPM || mo) cm.add8(m);
    }
    acc += ca.total() + 2 * cb.total() - 3 * cm.total();
  }
  if (acc == 0x12345678u) out[0] = acc;
}

// mode 5: k_site variant 0's per-population structure (47 + 32 + 1 pairs: batches of 8 + remainder loop with direct
// popcounts) and per-population totals, no shared memory, no epilogue
__global__ void __launch_bounds__(256, 4) k_pops(const uint2* __restrict__ p, int64_t n_tiles, int pps, uint32_t* out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t acc = 0;
  const int npairs[3] = {47, 32, 1};
  for (int64_t t = (int64_t)blockIdx.x * 8 + warp; t < n_tiles; t += (int64_t)gridDim.x * 8) {
    const uint2* tile = p + (size_t)t * pps * 32 + lane;
    int off = 0;
    for (int pi = 0; pi < 3; ++pi) {
      const uint2* col = tile + (size_t)off * 32;
      const int n = npairs[pi];
      off += n;
      SliceCounter ca, cb, cm;
      int q = 0;
      for (; q + 8 <= n; q += 8) {
        uint2 v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = ld_stream(col + (size_t)(q + i) * 32);
        uint32_t a[8], b[8], m[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) { a[i] = v[i].x; b[i] = v[i].y; m[i] = v[i].x & v[i].y; }
        ca.add8(a); cb.add8(b); cm.add8(m);
      }
      int aa = ca.total(), ab = cb.total(), am = cm.total();
#pragma unroll 4
      for (; q < n; ++q) {
        uint2 v = ld_stream(col + (size_t)q * 32);
        aa += __popc(v.x); ab += __popc(v.y); am += __popc(v.x & v.y);
      }
      acc += (aa + 2 * ab - 3 * am) * (pi + 1);
    }
  }
  if (acc == 0x12345678u) out[0] = acc;
}

__global__ void __launch_bounds__(256) k_one_pair(const uint2* __restrict__ p, int64_t n_tiles, int pps, uint32_t* out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t acc = 0;
  for (int64_t t0 = ((int64_t)blockIdx.x * 8 + warp) * 8; t0 < n_tiles; t0 += (int64_t)gridDim.x * 64) {
    uint2 v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
      v[i] = t0 + i < n_tiles ? ld_stream(p + ((size_t)(t0 + i) * pps + pps - 1) * 32 + lane) : make_uint2(0u, 0u);
#pragma unroll
    for (int i = 0; i < 8; ++i) acc ^= v[i].x ^ v[i].y;
  }
  if (acc == 0x12345678u) out[0] = acc;
}

int main(int argc, char** argv) {
  const int64_t n_sites = argc > 1 ? atoll(argv[1]) : 6000000;
  const int pps = argc > 2 ? atoi(argv[2]) : 80;
  const int64_t n_tiles = (n_sites + 31) / 32;
  const size_t bytes = (size_t)n_tiles * pps * 256;
  void* d;
  uint32_t* out;
  cudaMalloc(&d, bytes);
  cudaMalloc(&out, 4);
  cudaMemset(d, argc > 3 ? atoi(argv[3]) : 0x5a, bytes);
  int sms = 0;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0);
  cudaEvent_t a, b;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  for (int mode = 1; mode < 7; ++mode) {
    if (mode == 2 || mode == 4) continue;
    const size_t mode_bytes = mode == 6 ? (size_t)n_tiles * 256 : bytes;
    for (int bps : {3, 4}) {
      float best = 1e9f, sum = 0;
      const int reps = 12;
      for (int r = 0; r < reps + 3; ++r) {
        cudaEventRecord(a);
        if (mode == 0) k_flat<<<sms * bps, 256>>>((const uint4*)d, bytes / 16, out);
        else if (mode == 1) k_tiles<8><<<sms * bps, 256>>>((const uint2*)d, n_tiles, pps, out);
        else if (mode == 2) k_tiles<16><<<sms * bps, 256>>>((const uint2*)d, n_tiles, pps, out);
        else if (mode == 3) k_csa<false><<<sms * bps, 256>>>((const uint2*)d, n_tiles, pps, out);
        else if (mode == 4) k_csa<true><<<sms * bps, 256>>>((const uint2*)d, n_tiles, pps, out);
        else if (mode == 6) k_one_pair<<<sms * bps, 256>>>((const uint2*)d, n_tiles, pps, out);
        else k_pops<<<sms * bps, 256>>>((const uint2*)d, n_tiles, pps, out);
        cudaEventRecord(b);
        cudaEventSynchronize(b);
        float ms;
        cudaEventElapsedTime(&ms, a, b);
        if (r >= 3) { sum += ms; if (ms < best) best = ms; }
      }
      printf("{\"mode\": %d, \"blocks_per_sm\": %d, \"bytes\": %zu, \"ms_mean\": %.4f, \"ms_best\": %.4f, \"GBps_mean\": %.1f, \"GBps_best\": %.1f}\n",
             mode, bps, mode_bytes, sum / reps, best, mode_bytes / (sum / reps) / 1e6, mode_bytes / best / 1e6);
    }
  }
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { printf("error %s\n", cudaGetErrorString(e)); return 1; }
  return 0;
}
