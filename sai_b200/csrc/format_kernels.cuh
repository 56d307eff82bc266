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

int format_scores(FormatState& f, const sai_format_input* in, cudaStream_t st, int64_t* sizes);
int format_text(FormatState& f, int which, char* out, int64_t cap, cudaStream_t st);
int format_stats(FormatState& f, double* out, int n);
int format_doubles_device(const double* x, int64_t n, char* out, cudaStream_t st);
void format_release(FormatState& f);

}  // namespace sai
