// Shared helpers for the sai_b200 CUDA sources (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/sai_b200.h"

namespace sai {

void set_error(const char* fmt, ...);

#define SAI_CUDA_CHECK(expr)                                                        \
  do {                                                                              \
    cudaError_t _e = (expr);                                                        \
    if (_e != cudaSuccess) {                                                        \
      ::sai::set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #expr,           \
                       cudaGetErrorString(_e));                                     \
      return SAI_E_CUDA;                                                            \
    }                                                                               \
  } while (0)

#define SAI_REQUIRE(cond, ...)          \
  do {                                  \
    if (!(cond)) {                      \
      ::sai::set_error(__VA_ARGS__);    \
      return SAI_E_ARG;                 \
    }                                   \
  } while (0)

int validate_layout(const sai_layout* lay);
int validate_jobs(const sai_layout* lay, const sai_job* jobs, int32_t n_jobs);

// Number of SMs of the current device (cached per device).
int sm_count();

constexpr int kTile = SAI_TILE_SITES;  // sites per tile == warp width

// inflate_device.cu: sai_bgzf_inflate_device that also lowers *d_first_bad to first_index + i for
// every failed block i (d_first_bad may be NULL).
int bgzf_inflate_launch(const uint8_t* d_comp, const sai_bgzf_block* d_blocks, int64_t n_blocks, uint8_t* d_out,
                        int32_t* d_status, unsigned long long* d_first_bad, int64_t first_index, cudaStream_t stream);

// Kernel-parameter block shared by the site kernels (passed __grid_constant__).
struct JobBlock {
  int32_t n_jobs;
  int32_t pad_;
  sai_job job[SAI_MAX_JOBS];
};

}  // namespace sai
