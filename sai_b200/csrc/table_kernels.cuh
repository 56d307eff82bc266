// Outlier tables built from a score file on the device (table_kernels.cu): the engine's state.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/sai_b200.h"

namespace sai {

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
};

struct TableState {
  DevBuf text;        // the file, zero-padded to whole 16 KiB chunks
  DevBuf line;        // int64 [n_rows + 2]: byte offset of every line, + one past the last line's '\n'
  DevBuf cell;        // uint16 [n_rows][n_cols]: offset of every data cell within its line
  DevBuf cls;         // uint32 [n_chunks][n_cols]: OR of the cells' classes per pandas parse chunk
  DevBuf misc;        // flags, counters, small inputs and outputs
  DevBuf rows;        // per data row: chrom run scan, row text length, start, end
  DevBuf sort;        // sort keys and two permutations
  DevBuf lens;        // int64 [n_tables][n_rows + 1] + 1: table lengths, scanned to offsets
  DevBuf out;         // the tables' text
  int64_t n_bytes = 0, n_rows = 0, n_cols = 0, chunk_rows = 0, n_chunks = 0;
  int32_t kind[SAI_TABLE_MAX_COLS] = {};
  int32_t first_metric = 0, chrom = 0, start = 0, end = 0;
  double* vals = nullptr;  // caller's [n_metric][n_rows] float64 (device)
  int64_t n_runs = 0;
  bool parsed = false, ordered = false;
  int64_t out_size = 0;
  cudaEvent_t ev[12] = {};
  bool timed[6] = {};
};

int table_load(TableState& t, const char* text, int64_t n_bytes, int32_t n_cols, int64_t chunk_rows, int64_t* info,
               cudaStream_t st);
int table_classes(TableState& t, uint32_t* out, int64_t cap, cudaStream_t st);
int table_parse(TableState& t, const int32_t* kinds, int32_t first_metric, int32_t chrom, int32_t start, int32_t end,
                double* d_vals, double* first_val, int64_t* n_runs, cudaStream_t st);
int table_runs(TableState& t, int64_t* off, int64_t* len, int64_t cap, cudaStream_t st);
int table_order(TableState& t, const int32_t* run_rank, int64_t n_runs, cudaStream_t st);
int table_build(TableState& t, const double* thr, const int32_t* strict, int64_t* offsets, cudaStream_t st);
int table_text(TableState& t, char* out, int64_t cap, cudaStream_t st);
int table_stats(TableState& t, double* out, int n);
int parse_doubles_device(const char* text, const int64_t* offs, int64_t n, double* out, uint8_t* ok, cudaStream_t st);
void table_release(TableState& t);

}  // namespace sai
