// Device inflater for bgzip (BGZF) blocks: compressed members in HBM -> their text in HBM.
//
// One warp per block (inflate_device.cuh: the per-block decoder, also built for the host fuzz):
// the decode tables live in the warp's slice of shared memory, the bit reader and symbol loop are
// lane-uniform, stored runs and match copies are expanded by the whole warp, and the output goes
// straight to HBM -- a back-reference stays inside the block's own <= 64 KB, which L1 / L2 serve.
// The CRC-32 is computed by the warp over 32 parts of the output and combined in GF(2).  A block
// that does not decode to exactly its ISIZE bytes with a matching CRC gets a non-zero status and
// its output range is filled with '\n' (a parse that follows sees empty lines there); no other
// block's output is touched.
#include "common.cuh"
#include "inflate_device.cuh"

namespace sai {

namespace {

constexpr int kWarps = 8;  // blocks (warps) per CTA: 8 x 3.6 KB of tables

__global__ void __launch_bounds__(kWarps * 32) k_bgzf_inflate(const uint8_t* __restrict__ comp,
                                                               const sai_bgzf_block* __restrict__ blocks, int64_t n_blocks,
                                                               uint8_t* __restrict__ out, int32_t* __restrict__ status,
                                                               unsigned long long* first_bad, int64_t first_index) {
  __shared__ uint32_t crc_tab[256];
  __shared__ infl::Tables tabs[kWarps];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) crc_tab[i] = infl::crc_table_entry((uint32_t)i);
  __syncthreads();
  const int warp = threadIdx.x >> 5;
  const infl::Team t{(int)(threadIdx.x & 31), 32};
  const int64_t b = (int64_t)blockIdx.x * kWarps + warp;
  if (b >= n_blocks) return;
  const sai_bgzf_block d = blocks[b];
  uint8_t* o = out + d.text_off;
  const uint32_t isize = d.isize;
  int st = infl::inflate_block(comp + d.comp_off, d.comp_bytes, o, isize, tabs[warp], t);
  __syncwarp();
  if (st == infl::kOk) {
    uint32_t s = infl::crc_share(o, isize, crc_tab, t);
    for (int k = 16; k; k >>= 1) s ^= __shfl_xor_sync(0xffffffffu, s, k);
    if (infl::crc_finish(s, isize) != d.crc) st = infl::kBadCrc;
  }
  if (st != infl::kOk) {
    for (uint32_t k = t.lane; k < isize; k += 32) o[k] = '\n';
    if (t.lane == 0 && first_bad) atomicMin(first_bad, (unsigned long long)(first_index + b));
  }
  if (t.lane == 0) status[b] = st;
}

}  // namespace

int bgzf_inflate_launch(const uint8_t* d_comp, const sai_bgzf_block* d_blocks, int64_t n_blocks, uint8_t* d_out,
                        int32_t* d_status, unsigned long long* d_first_bad, int64_t first_index, cudaStream_t stream) {
  if (n_blocks == 0) return SAI_OK;
  const int64_t grid = (n_blocks + kWarps - 1) / kWarps;
  k_bgzf_inflate<<<(unsigned)grid, kWarps * 32, 0, stream>>>(d_comp, d_blocks, n_blocks, d_out, d_status, d_first_bad,
                                                               first_index);
  SAI_CUDA_CHECK(cudaGetLastError());
  return SAI_OK;
}

}  // namespace sai

extern "C" int sai_bgzf_inflate_device(const uint8_t* d_comp, const sai_bgzf_block* d_blocks, int64_t n_blocks,
                                       uint8_t* d_out, int32_t* d_status, void* stream) {
  SAI_REQUIRE(n_blocks >= 0 && n_blocks < (int64_t(1) << 40), "sai_bgzf_inflate_device: bad block count");
  SAI_REQUIRE(n_blocks == 0 || (d_comp && d_blocks && d_out && d_status), "sai_bgzf_inflate_device: NULL argument");
  return sai::bgzf_inflate_launch(d_comp, d_blocks, n_blocks, d_out, d_status, nullptr, 0,
                                  static_cast<cudaStream_t>(stream));
}
