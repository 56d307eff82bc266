// Score file text formatted on the device (format_kernels.cu): the engine's state for it.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/sai_b200.h"

namespace sai {

struct FormatState {
  void* in = nullptr;             // grow-only: the inputs of the last call
  size_t in_cap = 0;
  char* text[3] = {};             // grow-only: rows, .U.log, .Q.log
  size_t text_cap[3] = {};
  int64_t size[3] = {};           // bytes of each text of the last call
  cudaEvent_t ev[5] = {};         // copy start, copy end, lengths scanned, writes start, writes end
  bool timed = false;             // ev[] recorded by the last call
};

// Block-wide exclusive scan of one int64 per thread (blockDim.x a multiple of 32, at most 1024);
// *total = the block's sum.
__device__ inline int64_t block_excl_scan64(int64_t v, int64_t* total) {
  __shared__ int64_t warp_sum[32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int64_t x = v;
  for (int d = 1; d < 32; d <<= 1) {
    const int64_t y = __shfl_up_sync(0xffffffffu, x, d);
    if (lane >= d) x += y;
  }
  if (lane == 31) warp_sum[w] = x;
  __syncthreads();
  if (w == 0) {
    int64_t s = lane < nw ? warp_sum[lane] : 0;
    for (int d = 1; d < 32; d <<= 1) {
      const int64_t y = __shfl_up_sync(0xffffffffu, s, d);
      if (lane >= d) s += y;
    }
    if (lane < nw) warp_sum[lane] = s;
  }
  __syncthreads();
  const int64_t before = (w > 0 ? warp_sum[w - 1] : 0) + x - v;
  *total = warp_sum[nw - 1];
  __syncthreads();
  return before;
}

// v[0 .. n) -> exclusive offsets in place, v[n] = total (the three-kernel scan of vcf_device.cu's
// negative-value table, on int64); chunk: (n + 1023) / 1024 int64 of scratch
void scan_lengths(int64_t* v, int64_t n, int64_t* chunk, cudaStream_t st);
// blocks for a grid-stride launch over `items` items, per_block per block (1 .. 8 per SM)
int grid_for(int64_t items, int per_block);
// grows a device buffer to >= bytes (contents lost); SAI_OK or SAI_E_NOMEM / SAI_E_CUDA
int grow_dev(void** p, size_t* cap, size_t bytes);

int format_scores(FormatState& f, const sai_format_input* in, cudaStream_t st, int64_t* sizes);
int format_text(FormatState& f, int which, char* out, int64_t cap, cudaStream_t st);
int format_stats(FormatState& f, double* out, int n);
int format_doubles_device(const double* x, int64_t n, char* out, cudaStream_t st);
void format_release(FormatState& f);

}  // namespace sai
