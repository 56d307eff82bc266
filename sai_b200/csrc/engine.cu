// Host-buffer engine: what a reference-side `ChunkPreprocessor.run`
// (sai/preprocessors/chunk_preprocessor.py:105-147) calls once per chunk.
//
// The packed tiles are copied host->device in slices on a copy stream while the
// genotype pass (K1) of the previous slice runs on the compute stream; the
// window kernels run once all slices are flagged; results come back in one
// batch of device->host copies.  Device buffers are grow-only and reused across
// calls (one engine per GPU / per worker process).
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <array>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <tuple>
#include <vector>

#include "common.cuh"
#include "format_kernels.cuh"
#include "table_kernels.cuh"
#include "host_pack.h"
#include "vcf_genome.cuh"
#include "zt_format.cuh"
#include "zt_simd.h"

// Persistent host threads of the ingest session: a call hands out tasks [0, n) and returns once all
// of them have run (the caller works too).  Threads are created once per engine, not per slice.
struct StagePool {
  std::vector<std::thread> th;
  std::mutex mu;
  std::condition_variable wake, idle;
  const std::function<void(int64_t)>* job = nullptr;
  int64_t n_tasks = 0, finished = 0;
  std::atomic<int64_t> next{0};
  uint64_t gen = 0;
  int active = 0;  // workers inside a generation's task loop
  bool stop = false;

  void work_loop(int64_t n, const std::function<void(int64_t)>& f) {
    int64_t mine = 0;
    for (int64_t i = next.fetch_add(1); i < n; i = next.fetch_add(1), ++mine) f(i);
    std::lock_guard<std::mutex> lk(mu);
    finished += mine;
    if (finished == n_tasks) idle.notify_all();
  }
  void worker() {
    uint64_t seen = 0;
    std::unique_lock<std::mutex> lk(mu);
    for (;;) {
      wake.wait(lk, [&] { return stop || (gen != seen && job != nullptr); });
      if (stop) return;
      seen = gen;
      const auto* f = job;
      const int64_t n = n_tasks;
      ++active;
      lk.unlock();
      work_loop(n, *f);
      lk.lock();
      if (--active == 0) idle.notify_all();
    }
  }
  void run(int n_threads, int64_t n, const std::function<void(int64_t)>& f) {
    if (n <= 0) return;
    n_threads = std::max(1, n_threads);
    {
      std::unique_lock<std::mutex> lk(mu);
      while ((int)th.size() < n_threads - 1) th.emplace_back([this] { worker(); });
      job = &f;
      n_tasks = n;
      finished = 0;
      next.store(0);
      ++gen;
    }
    wake.notify_all();
    work_loop(n, f);
    std::unique_lock<std::mutex> lk(mu);
    // every task has run and no worker is still inside this generation's loop (it would take the
    // next generation's indices with this generation's job)
    idle.wait(lk, [&] { return finished == n_tasks && active == 0; });
    job = nullptr;
  }
  ~StagePool() {
    {
      std::lock_guard<std::mutex> lk(mu);
      stop = true;
    }
    wake.notify_all();
    for (auto& t : th) t.join();
  }
};

struct sai_engine {
  int device = 0;
  cudaStream_t s_copy = nullptr, s_comp = nullptr;
  std::vector<cudaEvent_t> ev;
  std::vector<cudaEvent_t> ev_dec;    // int8 pipeline, zt wire: slice decoded (its device ring slot is free again)
  int host_threads = 0;               // packer threads of the int8 pipeline (0: hardware concurrency)
  int i8_wire = 0;                    // wire format of the int8 pipeline: 0 = auto, 1 = dense tiles, 2 = zt records
  void* ring = nullptr;               // pinned staging ring of the int8 pipeline
  size_t ring_cap = 0;
  void* h_ztoff = nullptr;            // pinned tile directory of the int8 pipeline's zt records
  size_t h_ztoff_cap = 0;
  uint64_t i8_wire_bytes = 0;         // bytes the last int8 call put on the wire (tiles only)
  // grow-only device buffers
  struct Buf {
    void* p = nullptr;
    size_t cap = 0;
  };
  Buf packed, pos, win, mask, qval, res, cand, counts, sums, hist, neg, dd, zt, ztoff;
  // state of the last call (for sai_engine_rescore_windows)
  int64_t n_sites = 0, W = 0;
  int32_t n_jobs = 0;
  sai_job jobs[SAI_MAX_JOBS];
  sai_layout lay{};  // layout of the resident tiles (sai_engine_score_resident)
  // sai_engine_score_loaded_pieces: (first window, windows, first site, sites) per piece; empty = one chunk.
  // Per-window first / last sites follow the window bounds in `win`.
  std::vector<std::array<int64_t, 4>> pieces;
  // ingest session (sai_engine_vcf_*): text ring (pinned + device), the query and its tables
  struct Vcf {
    int state = 0;                    // 0 none, 1 feeding, 2 finished (tiles resident)
    sai_vcf_query q{};
    bool genome = false;              // sai_engine_vcf_genome_begin: the chromosome table of gq
    sai::VcfGenomeQuery gq{};
    int64_t site_cap = 0;             // sites the tile / position buffers hold (multiple of 32)
    int64_t row_bytes = 64;           // lower bound of a record's length: sizes the tile buffer
    int64_t fed = 0, n_slices = 0;
    int64_t slice_bytes = 32ll << 20; // sai_engine_set_vcf_slicing
    int ring = 4;
    size_t slot_bytes = 0;            // capacity of one ring slot (pinned and device)
    char* h_ring = nullptr;
    std::vector<cudaEvent_t> copied, parsed;  // per slot: H2D done (host slot free), parse done (device slot free)
    // per slice: H2D start / end, parse start / end, device inflate start / end (stage timing)
    std::vector<std::array<cudaEvent_t, 6>> tev;
    std::vector<char> inflated;       // per slice: its text was inflated on the device
    std::vector<char> carry;          // bgzip feed: the incomplete line at the end of the last slot
    double t_stage = 0, t_wait = 0;   // host seconds: staging / inflating into the ring, waiting for a free slot
    double t_launch = 0, t_feed = 0;  // host seconds: enqueueing copies and kernels, inside the feed calls
    double t_boundary = 0;            // host seconds inflating the boundary blocks of device-inflated groups
    double comp_bytes = 0;            // compressed bytes (with descriptors) copied for device inflate
    char* h_comp = nullptr;           // pinned ring of compressed groups (device inflate), comp_slot bytes a slot
    size_t comp_slot = 0;             // 0: (re)built by the next device-inflated group, for `ring` slots
    std::vector<cudaStream_t> s_infl; // per ring slot: the stream its inflates run on (slices inflate side by side)
    double stats[14] = {0};           // sai_engine_vcf_stats of the last finished session
    int sticky_rc = SAI_OK;           // first failure of the session, reported by finish
    StagePool pool;
    // negative-value table (DD): sai_engine_set_vcf_neg_table, then per session
    bool neg_on = false;              // the sessions that follow keep the table
    int64_t neg_min = 0;              // lower bound of its capacity (a repeat after SAI_E_CAPACITY)
    bool neg = false;                 // the current / last session keeps it
    sai::VcfNegSession negs{};        // its device buffers (vneg, vnega)
    int64_t neg_n = -1;               // entries the last finished session found (-1: none)
    std::vector<int64_t> neg_off;     // [n_chrom][n_pops + 1] offsets of the finished table (vnegt)
    std::vector<std::array<int64_t, 2>> chrom_sites;  // genome session: (first site, sites) per chromosome
  } vcf;
  Buf vtext, vscratch, vcols, vanc_pos, vanc_all, vstate;
  Buf vcomp, vbad;  // device inflate: ring of compressed groups (+ block statuses), first corrupt block
  Buf vgen;         // genome ingest: hash table, names, offsets, running state, per-chromosome records
  Buf vneg, vnega, vnegt;  // negative-value table: state + per-key counts, appended entries, finished table
  sai::FormatState fmt;    // score file text (sai_engine_format_scores)
  sai::TableState tab;     // outlier tables (sai_engine_table_*)
};

namespace sai {

static int grow(sai_engine::Buf& b, size_t bytes) {
  if (bytes <= b.cap) return SAI_OK;
  if (b.p) SAI_CUDA_CHECK(cudaFree(b.p));
  b.p = nullptr;
  b.cap = 0;
  const size_t want = bytes + bytes / 8 + 256;
  cudaError_t e = cudaMalloc(&b.p, want);
  if (e != cudaSuccess) {
    set_error("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
    return SAI_E_NOMEM;
  }
  b.cap = want;
  return SAI_OK;
}

static inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }

struct ResLayout {
  size_t nsnps, u, q, q_cnt, u_start, q_start, totals, total;
};
static ResLayout res_layout(int64_t W, int n_jobs) {
  ResLayout r{};
  size_t at = 0;
  const size_t n = (size_t)n_jobs * (size_t)W;
  r.nsnps = at, at += align256(sizeof(int32_t) * n);
  r.u = at, at += align256(sizeof(int64_t) * n);
  r.q = at, at += align256(sizeof(double) * n);
  r.q_cnt = at, at += align256(sizeof(int32_t) * n);
  r.u_start = at, at += align256(sizeof(int64_t) * n);
  r.q_start = at, at += align256(sizeof(int64_t) * n);
  r.totals = at, at += align256(sizeof(int64_t) * 2 * n_jobs);
  r.total = at;
  return r;
}

// The pieces the resident tiles were scored in: those of sai_engine_score_loaded_pieces, or one chunk as
// the one piece (0, W, 0, n_sites).
static std::vector<std::array<int64_t, 4>> scored_pieces(const sai_engine* e) {
  if (!e->pieces.empty()) return e->pieces;
  return {{0, e->W, 0, e->n_sites}};
}

// Window kernel on the device-resident flags + results back to the host.
static int run_windows(sai_engine* e, sai_host_results* out) {
  const int64_t W = e->W;
  const int n_jobs = e->n_jobs;
  const int64_t n_tiles = sai_num_tiles(e->n_sites);
  const int64_t stride = n_tiles * kTile;
  const ResLayout rl = res_layout(W, n_jobs);
  const size_t cu = align256(sizeof(int32_t) * (size_t)n_jobs * out->cap_u);
  const size_t cq = align256(sizeof(int32_t) * (size_t)n_jobs * out->cap_q);
  if (int rc = grow(e->cand, cu + cq + 256)) return rc;
  char* res = static_cast<char*>(e->res.p);
  const uint32_t* d_mask_u = static_cast<const uint32_t*>(e->mask.p);
  const uint32_t* d_mask_q = d_mask_u + (size_t)n_jobs * n_tiles;
  const int64_t* d_ws = static_cast<const int64_t*>(e->win.p);
  int32_t* d_uc = static_cast<int32_t*>(e->cand.p);
  int32_t* d_qc = reinterpret_cast<int32_t*>(static_cast<char*>(e->cand.p) + cu);
  cudaStream_t st = e->s_comp;
  const int32_t* d_first = reinterpret_cast<const int32_t*>(d_ws + 2 * W);
  if (int rc = e->pieces.empty()
                   ? sai_window_stats(
                         static_cast<const int32_t*>(e->pos.p), e->n_sites, d_ws, d_ws + W, W, e->jobs, n_jobs,
                         d_mask_u, d_mask_q, static_cast<const double*>(e->qval.p), stride,
                         reinterpret_cast<int32_t*>(res + rl.nsnps), reinterpret_cast<int64_t*>(res + rl.u),
                         reinterpret_cast<double*>(res + rl.q), reinterpret_cast<int32_t*>(res + rl.q_cnt),
                         reinterpret_cast<int64_t*>(res + rl.u_start), reinterpret_cast<int64_t*>(res + rl.q_start),
                         reinterpret_cast<int64_t*>(res + rl.totals), d_uc, out->cap_u, d_qc, out->cap_q, st)
                   : sai_window_stats_pieces(
                         static_cast<const int32_t*>(e->pos.p), e->n_sites, d_ws, d_ws + W, d_first, d_first + W, W,
                         e->jobs, n_jobs, d_mask_u, d_mask_q, static_cast<const double*>(e->qval.p), stride,
                         reinterpret_cast<int32_t*>(res + rl.nsnps), reinterpret_cast<int64_t*>(res + rl.u),
                         reinterpret_cast<double*>(res + rl.q), reinterpret_cast<int32_t*>(res + rl.q_cnt),
                         reinterpret_cast<int64_t*>(res + rl.u_start), reinterpret_cast<int64_t*>(res + rl.q_start),
                         reinterpret_cast<int64_t*>(res + rl.totals), d_uc, out->cap_u, d_qc, out->cap_q, st))
    return rc;
  const size_t n = (size_t)n_jobs * (size_t)W;
  if (n > 0) {
    SAI_CUDA_CHECK(cudaMemcpyAsync(out->nsnps, res + rl.nsnps, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, st));
    SAI_CUDA_CHECK(cudaMemcpyAsync(out->u, res + rl.u, sizeof(int64_t) * n, cudaMemcpyDeviceToHost, st));
    SAI_CUDA_CHECK(cudaMemcpyAsync(out->q, res + rl.q, sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    SAI_CUDA_CHECK(cudaMemcpyAsync(out->q_cnt, res + rl.q_cnt, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, st));
    SAI_CUDA_CHECK(cudaMemcpyAsync(out->u_start, res + rl.u_start, sizeof(int64_t) * n, cudaMemcpyDeviceToHost, st));
    SAI_CUDA_CHECK(cudaMemcpyAsync(out->q_start, res + rl.q_start, sizeof(int64_t) * n, cudaMemcpyDeviceToHost, st));
  }
  SAI_CUDA_CHECK(cudaMemcpyAsync(out->totals, res + rl.totals, sizeof(int64_t) * 2 * n_jobs, cudaMemcpyDeviceToHost, st));
  SAI_CUDA_CHECK(cudaStreamSynchronize(st));
  bool fits = true;
  for (int j = 0; j < n_jobs; ++j) {
    const int64_t tu = out->totals[2 * j], tq = out->totals[2 * j + 1];
    if (tu > out->cap_u || tq > out->cap_q) {
      fits = false;
      continue;
    }
    if (tu > 0)
      SAI_CUDA_CHECK(cudaMemcpyAsync(out->u_cand + (size_t)j * out->cap_u, d_uc + (size_t)j * out->cap_u,
                                     sizeof(int32_t) * tu, cudaMemcpyDeviceToHost, st));
    if (tq > 0)
      SAI_CUDA_CHECK(cudaMemcpyAsync(out->q_cand + (size_t)j * out->cap_q, d_qc + (size_t)j * out->cap_q,
                                     sizeof(int32_t) * tq, cudaMemcpyDeviceToHost, st));
  }
  SAI_CUDA_CHECK(cudaStreamSynchronize(st));
  if (!fits) {
    set_error("candidate capacity too small (see totals)");
    return SAI_E_CAPACITY;
  }
  return SAI_OK;
}

static int check_results(const sai_host_results* out) {
  SAI_REQUIRE(out && out->nsnps && out->u && out->q && out->q_cnt && out->u_start && out->q_start &&
                  out->totals,
              "NULL result pointer");
  SAI_REQUIRE(out->cap_u >= 0 && out->cap_q >= 0 && (out->cap_u == 0 || out->u_cand) &&
                  (out->cap_q == 0 || out->q_cand),
              "bad candidate buffers");
  return SAI_OK;
}

}  // namespace sai

using namespace sai;

extern "C" {

int sai_engine_create(int32_t device, sai_engine** out) {
  SAI_REQUIRE(out, "NULL argument");
  SAI_CUDA_CHECK(cudaSetDevice(device));
  sai_engine* e = new sai_engine();
  e->device = device;
  SAI_CUDA_CHECK(cudaStreamCreateWithFlags(&e->s_copy, cudaStreamNonBlocking));
  SAI_CUDA_CHECK(cudaStreamCreateWithFlags(&e->s_comp, cudaStreamNonBlocking));
  *out = e;
  return SAI_OK;
}

void sai_engine_destroy(sai_engine* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  for (auto* b : {&e->packed, &e->pos, &e->win, &e->mask, &e->qval, &e->res, &e->cand, &e->counts, &e->sums, &e->hist,
                  &e->neg, &e->dd, &e->zt, &e->ztoff, &e->vtext, &e->vscratch, &e->vcols, &e->vanc_pos, &e->vanc_all,
                  &e->vstate, &e->vcomp, &e->vbad})
    if (b->p) cudaFree(b->p);
  for (auto ev : e->ev) cudaEventDestroy(ev);
  for (auto ev : e->ev_dec) cudaEventDestroy(ev);
  for (auto ev : e->vcf.copied) cudaEventDestroy(ev);
  for (auto ev : e->vcf.parsed) cudaEventDestroy(ev);
  for (auto& t : e->vcf.tev)
    for (auto ev : t) cudaEventDestroy(ev);
  if (e->vcf.h_ring) cudaFreeHost(e->vcf.h_ring);
  if (e->vcf.h_comp) cudaFreeHost(e->vcf.h_comp);
  for (auto s : e->vcf.s_infl) cudaStreamDestroy(s);
  if (e->ring) cudaFreeHost(e->ring);
  if (e->h_ztoff) cudaFreeHost(e->h_ztoff);
  sai::format_release(e->fmt);
  sai::table_release(e->tab);
  if (e->s_copy) cudaStreamDestroy(e->s_copy);
  if (e->s_comp) cudaStreamDestroy(e->s_comp);
  delete e;
}

// int8 pipeline (sai_engine_score_host_i8): the reference-side representation -- one int8 matrix
// of per-individual allele sums per population, pageable host memory -- is packed into tiled
// bit-planes by a pool of host threads, slice by slice, straight into a ring of pinned staging
// buffers; as soon as a slice is complete it goes H2D and, once landed, through the genotype
// pass, while the threads are already packing the following slices.  Three stages overlap: pack
// (host cores, reads 4x the bytes it writes) | PCIe copy | K1.
//
// Wire format (sai_engine_set_i8_wire).  The packers saturate the host's memory system, so every
// byte they do not write -- and the copy engine does not read back -- is throughput.  By default a
// packer keeps the tile it has just packed in its L1, turns it into a zt record on the spot
// (zt_simd.cpp) and streams the records of its block of tiles, back to back, to the block's fixed
// region of the ring slot (region = where the dense tiles would have gone, so no packer waits for
// another one's length).  A slice then goes out as ONE strided copy (rows = blocks, width = the
// longest block) into a device ring laid out like the pinned one, followed by the slice's part of
// the tile directory; k_zt_decode rebuilds the dense tiles in HBM in front of K1 and frees the
// device slot.
struct I8Source {
  const int8_t* const* gt;
  const int64_t* row_stride;
};

static int stream_tiles_from_i8(sai_engine* e, const sai_layout* lay, const I8Source& src, int64_t n_sites,
                                int64_t n_tiles, const sai_job* jobs, int32_t n_jobs, uint32_t* d_mask_u,
                                uint32_t* d_mask_q, double* d_qval, int64_t stride) {
  const size_t tile_bytes = (size_t)lay->pairs_per_site * kTile * 8;
  uint64_t slice_bytes = 32ull << 20;
  int kRing = 4;
#ifdef SAI_EXPERIMENTS
  if (const char* v = getenv("SAI_I8_SLICE_MB")) slice_bytes = (uint64_t)std::max(1, atoi(v)) << 20;  // tools/ A/B knobs
  if (const char* v = getenv("SAI_I8_RING")) kRing = std::max(2, atoi(v));
#endif
  // a small chunk does not need (or pay for) the full ring: at most n_tiles / kRing tiles per slot
  const int64_t slice_tiles = std::max<int64_t>(1, std::min<int64_t>((int64_t)(slice_bytes / tile_bytes), (n_tiles + kRing - 1) / kRing));
  const int64_t n_slices = (n_tiles + slice_tiles - 1) / slice_tiles;
  const size_t slot_bytes = (size_t)slice_tiles * tile_bytes;
  if (e->ring_cap < slot_bytes * kRing) {
    if (e->ring) SAI_CUDA_CHECK(cudaFreeHost(e->ring));
    e->ring = nullptr;
    e->ring_cap = 0;
    SAI_CUDA_CHECK(cudaHostAlloc(&e->ring, slot_bytes * kRing, cudaHostAllocDefault));
    e->ring_cap = slot_bytes * kRing;
  }
  while ((int64_t)e->ev.size() < kRing) {
    cudaEvent_t ev;
    SAI_CUDA_CHECK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    e->ev.push_back(ev);
  }
  // auto: zt records when this CPU has the vector record encoder (the portable one would be the bottleneck)
  const bool zt = e->i8_wire == 2 || (e->i8_wire == 0 && strcmp(zt_isa(), "portable") != 0);
  const int P = lay->pairs_per_site;
  std::vector<uint64_t> padc(P);
  uint64_t* h_off = nullptr;
  if (zt) {
    for (int r = 0; r < P; ++r) padc[r] = pad_constant(*lay, r);
    const size_t need = sizeof(uint64_t) * (size_t)(n_tiles + 1);
    if (e->h_ztoff_cap < need) {
      if (e->h_ztoff) SAI_CUDA_CHECK(cudaFreeHost(e->h_ztoff));
      e->h_ztoff = nullptr;
      e->h_ztoff_cap = 0;
      SAI_CUDA_CHECK(cudaHostAlloc(&e->h_ztoff, need + need / 4, cudaHostAllocDefault));
      e->h_ztoff_cap = need + need / 4;
    }
    h_off = static_cast<uint64_t*>(e->h_ztoff);
    // the records live in a device ring laid out like the pinned one: a slot is rewritten once its
    // slice has been decoded (ev_dec)
    if (int k = grow(e->zt, slot_bytes * kRing + 256)) return k;
    if (int k = grow(e->ztoff, need + 256)) return k;
    while ((int64_t)e->ev_dec.size() < kRing) {
      cudaEvent_t ev;
      SAI_CUDA_CHECK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
      e->ev_dec.push_back(ev);
    }
  }
  int n_threads = e->host_threads > 0 ? e->host_threads : (int)std::max(1u, std::thread::hardware_concurrency());
  // packing tasks: blocks of tiles, in slice order
  int64_t block_cap = 32;
#ifdef SAI_EXPERIMENTS
  if (const char* v = getenv("SAI_I8_BLOCK_TILES")) block_cap = std::max(1, atoi(v));
#endif
  const int64_t block_tiles = std::max<int64_t>(1, std::min<int64_t>(block_cap, (slice_tiles + 2 * n_threads - 1) / (2 * n_threads)));
  const int64_t blocks_per_slice = (slice_tiles + block_tiles - 1) / block_tiles;
  auto blocks_of = [&](int64_t s) {
    const int64_t tiles = std::min(slice_tiles, n_tiles - s * slice_tiles);
    return (tiles + block_tiles - 1) / block_tiles;
  };
  const int64_t n_tasks = (n_slices - 1) * blocks_per_slice + blocks_of(n_slices - 1);
  n_threads = (int)std::min<int64_t>(n_threads, n_tasks);
  std::unique_ptr<uint32_t[]> used(new uint32_t[n_tasks]);  // zt: bytes of block i's records (whole 64-byte lines)
  std::atomic<uint64_t> wire_bytes{0};
  std::atomic<int64_t> next_task{0};
  std::unique_ptr<std::atomic<int>[]> done(new std::atomic<int>[n_slices]);
  for (int64_t s = 0; s < n_slices; ++s) done[s].store(0);
  std::atomic<int> bad{0}, abort_flag{0};
  uint8_t* ring = static_cast<uint8_t*>(e->ring);
  // Slices are handed to the GPU by whichever packer thread completes them (in slice order, under
  // issue_mu): no hand-off to a feeding thread, so no wake-up latency between "packed" and "on the
  // wire", and nothing but copies in the copy stream (a host callback there would stall the next
  // copy until a CPU is free to run it -- all of them are packing).  A ring slot is free again when
  // the copy event of the slice that used it last has completed; the packers check that themselves
  // (`slot_free`), which in the pack-bound steady state is a single relaxed load.
  std::mutex issue_mu;
  int64_t next_issue = 0;          // guarded by issue_mu
  std::atomic<int64_t> issued{0};  // == next_issue, readable without the lock
  std::atomic<int64_t> freed{0};   // copies [0, freed) have left their ring slots
  std::mutex free_mu;
  int rc = SAI_OK;      // guarded by issue_mu
  std::string err_msg;  // the failing thread's message (sai_last_error is thread-local)
  auto fail_locked = [&](int code) {
    if (rc == SAI_OK) {
      rc = code;
      err_msg = sai_last_error();
    }
    abort_flag.store(1);
  };
  auto slot_free = [&](int64_t s) {  // may slice s be packed into its ring slot?
    if (s < kRing || freed.load(std::memory_order_acquire) > s - kRing) return true;
    std::lock_guard<std::mutex> lk(free_mu);
    int64_t f = freed.load(std::memory_order_relaxed);
    // the event of slot f % kRing still belongs to slice f: slice f + kRing is not packed before f is freed
    while (f < issued.load(std::memory_order_acquire) && cudaEventQuery(e->ev[f % kRing]) == cudaSuccess) ++f;
    freed.store(f, std::memory_order_release);
    return f > s - kRing;
  };
  auto issue_ready_slices = [&]() {
    std::lock_guard<std::mutex> lk(issue_mu);
    while (rc == SAI_OK && next_issue < n_slices &&
           done[next_issue].load(std::memory_order_acquire) == (int)blocks_of(next_issue)) {
      const int64_t s = next_issue;
      if (bad.load()) {
        fail_locked(SAI_E_DOMAIN);
        break;
      }
      const int64_t t0 = s * slice_tiles, t1 = std::min(n_tiles, t0 + slice_tiles);
      const int slot = (int)(s % kRing);
      cudaError_t ce = cudaSuccess;
      if (!zt) {
        ce = cudaMemcpyAsync(static_cast<char*>(e->packed.p) + (size_t)t0 * tile_bytes, ring + (size_t)slot * slot_bytes,
                             (size_t)(t1 - t0) * tile_bytes, cudaMemcpyHostToDevice, e->s_copy);
        wire_bytes.fetch_add((uint64_t)(t1 - t0) * tile_bytes, std::memory_order_relaxed);
      } else {
        // rows = the slice's blocks (pitch = a block's dense size), width = the longest record run;
        // a shorter last block goes separately so that no row reaches past the slot
        const int64_t nb = blocks_of(s), task0 = s * blocks_per_slice;
        const bool short_last = (t1 - t0) % block_tiles != 0;
        const int64_t rows = short_last ? nb - 1 : nb;
        const size_t pitch = (size_t)block_tiles * tile_bytes;
        size_t width = 0;
        for (int64_t b = 0; b < rows; ++b) width = std::max<size_t>(width, used[task0 + b]);
        char* dst = static_cast<char*>(e->zt.p) + (size_t)slot * slot_bytes;
        const uint8_t* srcp = ring + (size_t)slot * slot_bytes;
        if (s >= kRing) ce = cudaStreamWaitEvent(e->s_copy, e->ev_dec[slot], 0);  // the slot's previous slice is decoded
        if (ce == cudaSuccess && rows > 0 && width > 0)
          ce = cudaMemcpy2DAsync(dst, pitch, srcp, pitch, width, (size_t)rows, cudaMemcpyHostToDevice, e->s_copy);
        if (ce == cudaSuccess && short_last && used[task0 + nb - 1] > 0)
          ce = cudaMemcpyAsync(dst + (size_t)rows * pitch, srcp + (size_t)rows * pitch, used[task0 + nb - 1],
                               cudaMemcpyHostToDevice, e->s_copy);
        if (ce == cudaSuccess)
          ce = cudaMemcpyAsync(static_cast<uint64_t*>(e->ztoff.p) + t0, h_off + t0, sizeof(uint64_t) * (size_t)(t1 - t0),
                               cudaMemcpyHostToDevice, e->s_copy);
        wire_bytes.fetch_add((uint64_t)width * rows + (short_last ? used[task0 + nb - 1] : 0) + 8ull * (t1 - t0),
                             std::memory_order_relaxed);
      }
      if (ce == cudaSuccess) ce = cudaEventRecord(e->ev[slot], e->s_copy);
      if (ce == cudaSuccess) ce = cudaStreamWaitEvent(e->s_comp, e->ev[slot], 0);
      if (ce != cudaSuccess) {
        set_error("int8 pipeline: CUDA call failed: %s", cudaGetErrorString(ce));
        fail_locked(SAI_E_CUDA);
        break;
      }
      ++next_issue;
      issued.store(next_issue, std::memory_order_release);
      if (zt) {
        int k = sai_zt_decode(lay, e->zt.p, (uint64_t)slot_bytes * kRing, static_cast<const uint64_t*>(e->ztoff.p), t0, t1 - t0,
                              e->packed.p, e->s_comp);
        if (k == SAI_OK && cudaEventRecord(e->ev_dec[slot], e->s_comp) != cudaSuccess) {
          set_error("int8 pipeline: cudaEventRecord failed");
          k = SAI_E_CUDA;
        }
        if (k) {
          fail_locked(k);
          break;
        }
      }
      if (int k = sai_site_flags(lay, e->packed.p, t0, t1 - t0, n_tiles, jobs, n_jobs, d_mask_u, d_mask_q, d_qval,
                                 stride, nullptr, nullptr, 0, 0, e->s_comp))
        fail_locked(k);
    }
  };
  const int device = e->device;
  auto worker = [&]() {
    cudaSetDevice(device);  // a fresh thread starts on device 0
    std::unique_ptr<ZtBlockScratch> scratch(zt ? new ZtBlockScratch(P) : nullptr);
    for (;;) {
      const int64_t i = next_task.fetch_add(1);
      if (i >= n_tasks) break;
      const int64_t s = i / blocks_per_slice, b = i % blocks_per_slice;
      while (!slot_free(s) && !abort_flag.load())  // the slot's previous slice is still on the wire (rare:
        std::this_thread::sleep_for(std::chrono::microseconds(50));  // the copy is faster than the packers)
      if (abort_flag.load()) break;
      const int64_t t0 = s * slice_tiles + b * block_tiles;
      const int64_t t1 = std::min(std::min(n_tiles, (s + 1) * slice_tiles), t0 + block_tiles);
      uint8_t* slot = ring + (size_t)(s % kRing) * slot_bytes;
      if (zt) {
        // the block's records -> its region of the ring slot (= where its dense tiles would go); the device
        // ring is laid out like the pinned one, so a record's device offset is its offset in the ring
        uint8_t* region = slot + (size_t)(t0 - s * slice_tiles) * tile_bytes;
        bool bad_here = false;
        used[i] = (uint32_t)zt_pack_block_i8(*lay, src.gt, src.row_stride, n_sites, t0, t1, padc.data(), region,
                                             (uint64_t)(region - ring), h_off, *scratch, true, &bad_here);
        if (bad_here) bad.store(1);
      } else if (pack_tiles_i8_all(*lay, src.gt, src.row_stride, n_sites, t0, t1, s * slice_tiles, slot, 0)) {
        bad.store(1);
      }
      if (done[s].fetch_add(1, std::memory_order_acq_rel) + 1 == (int)blocks_of(s)) issue_ready_slices();
    }
  };
  std::vector<std::thread> pool;
  for (int i = 0; i < n_threads; ++i) pool.emplace_back(worker);
  for (auto& t : pool) t.join();
  issue_ready_slices();  // nothing left unless a packer bailed out
  const cudaError_t drained = cudaStreamSynchronize(e->s_copy);  // the ring may be reused by the next call
  e->i8_wire_bytes = wire_bytes.load();
  if (rc == SAI_E_DOMAIN || (rc == SAI_OK && bad.load())) {
    set_error("a genotype value does not fit the bit-planes of its population");
    return SAI_E_DOMAIN;
  }
  if (rc == SAI_OK && drained != cudaSuccess) {
    set_error("cudaStreamSynchronize failed: %s", cudaGetErrorString(drained));
    return SAI_E_CUDA;
  }
  if (rc != SAI_OK) set_error("%s", err_msg.c_str());
  return rc;
}

// Shared body of the host entry points: `packed` (dense tiles), the zero-suppressed stream +
// its tile directory when `zt_stream` is given, or int8 matrices (`i8`).
static int score_host_impl(sai_engine* e, const sai_layout* lay, const uint8_t* packed,
                           const uint8_t* zt_stream, const uint64_t* zt_off, const I8Source* i8, const int32_t* pos,
                           int64_t n_sites, const int64_t* win_start, const int64_t* win_end,
                           int64_t n_windows, const sai_job* jobs, int32_t n_jobs, sai_host_results* out) {
  SAI_REQUIRE(e, "NULL engine");
  if (int rc = validate_layout(lay)) return rc;
  if (int rc = validate_jobs(lay, jobs, n_jobs)) return rc;
  SAI_REQUIRE(n_sites >= 0 && n_windows >= 0, "negative size");
  SAI_REQUIRE(n_sites == 0 || ((packed || (zt_stream && zt_off) || i8) && pos), "NULL input");
  SAI_REQUIRE(n_windows == 0 || (win_start && win_end), "NULL windows");
  if (int rc = check_results(out)) return rc;
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  e->vcf.state = 0;  // the tiles of an ingest session are replaced
  const int64_t W = n_windows;
  const int64_t n_tiles = sai_num_tiles(n_sites);
  const int64_t stride = n_tiles * kTile;
  const size_t packed_bytes = sai_packed_bytes(lay, n_sites);
  const ResLayout rl = res_layout(W, n_jobs);
  const bool zt = zt_stream != nullptr && n_sites > 0;
  const uint64_t kRaw = 1ull << 63;
  const uint64_t zt_bytes = zt ? (zt_off[n_tiles] & ~kRaw) : 0;

  if (int rc = grow(e->packed, packed_bytes + 256)) return rc;
  if (int rc = grow(e->pos, sizeof(int32_t) * (size_t)stride + 256)) return rc;
  if (int rc = grow(e->win, sizeof(int64_t) * 2 * (size_t)W + 256)) return rc;
  if (int rc = grow(e->mask, sizeof(uint32_t) * 2 * (size_t)n_jobs * n_tiles + 256)) return rc;
  if (int rc = grow(e->qval, sizeof(double) * (size_t)n_jobs * stride + 256)) return rc;
  if (int rc = grow(e->res, rl.total + 256)) return rc;
  if (zt) {
    if (int rc = grow(e->zt, zt_bytes + 256)) return rc;
    if (int rc = grow(e->ztoff, sizeof(uint64_t) * (size_t)(n_tiles + 1) + 256)) return rc;
  }
  e->n_sites = n_sites;
  e->W = W;
  e->pieces.clear();
  e->n_jobs = n_jobs;
  e->lay = *lay;
  for (int j = 0; j < n_jobs; ++j) e->jobs[j] = jobs[j];

  uint32_t* d_mask_u = static_cast<uint32_t*>(e->mask.p);
  uint32_t* d_mask_q = d_mask_u + (size_t)n_jobs * n_tiles;
  double* d_qval = static_cast<double*>(e->qval.p);
  int32_t* d_pos = static_cast<int32_t*>(e->pos.p);
  int64_t* d_ws = static_cast<int64_t*>(e->win.p);

  // small inputs first
  if (n_sites > 0)
    SAI_CUDA_CHECK(cudaMemcpyAsync(d_pos, pos, sizeof(int32_t) * n_sites, cudaMemcpyHostToDevice, e->s_copy));
  if (W > 0) {
    SAI_CUDA_CHECK(cudaMemcpyAsync(d_ws, win_start, sizeof(int64_t) * W, cudaMemcpyHostToDevice, e->s_copy));
    SAI_CUDA_CHECK(cudaMemcpyAsync(d_ws + W, win_end, sizeof(int64_t) * W, cudaMemcpyHostToDevice, e->s_copy));
  }
  if (zt)
    SAI_CUDA_CHECK(cudaMemcpyAsync(e->ztoff.p, zt_off, sizeof(uint64_t) * (size_t)(n_tiles + 1),
                                   cudaMemcpyHostToDevice, e->s_copy));
  if (i8 && n_tiles > 0) {
    if (int rc = stream_tiles_from_i8(e, lay, *i8, n_sites, n_tiles, jobs, n_jobs, d_mask_u, d_mask_q, d_qval, stride))
      return rc;
    while (e->ev.empty()) {
      cudaEvent_t ev;
      SAI_CUDA_CHECK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
      e->ev.push_back(ev);
    }
    SAI_CUDA_CHECK(cudaEventRecord(e->ev[0], e->s_copy));  // positions / windows went on the copy stream
    SAI_CUDA_CHECK(cudaStreamWaitEvent(e->s_comp, e->ev[0], 0));
    return run_windows(e, out);
  }
  // sliced H2D of the tiles (about 32 MB on the wire per slice); per slice, as soon as it has
  // landed: [zt: rebuild the dense tiles,] then K1
  const size_t tile_bytes = (size_t)lay->pairs_per_site * kTile * 8;
  const uint64_t slice_bytes = 32ull << 20;
  std::vector<int64_t> cut{0};
  if (!zt) {
    const int64_t slice_tiles = std::max<int64_t>(1, (int64_t)(slice_bytes / tile_bytes));
    for (int64_t t = slice_tiles; t < n_tiles; t += slice_tiles) cut.push_back(t);
  } else {
    uint64_t start = 0;
    for (int64_t t = 1; t < n_tiles; ++t) {
      const uint64_t o = zt_off[t] & ~kRaw;
      SAI_REQUIRE(o >= (zt_off[t - 1] & ~kRaw) && o <= zt_bytes, "zt tile directory is not monotonic");
      if (o - start >= slice_bytes) {
        cut.push_back(t);
        start = o;
      }
    }
  }
  if (n_tiles > 0) cut.push_back(n_tiles);
  const int64_t n_slices = (int64_t)cut.size() - 1;
  while ((int64_t)e->ev.size() < n_slices + 1) {
    cudaEvent_t ev;
    SAI_CUDA_CHECK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    e->ev.push_back(ev);
  }
  for (int64_t s = 0; s < n_slices; ++s) {
    const int64_t t0 = cut[s], t1 = cut[s + 1];
    if (!zt) {
      SAI_CUDA_CHECK(cudaMemcpyAsync(static_cast<char*>(e->packed.p) + t0 * tile_bytes,
                                     packed + t0 * tile_bytes, (size_t)(t1 - t0) * tile_bytes,
                                     cudaMemcpyHostToDevice, e->s_copy));
    } else {
      const uint64_t b0 = zt_off[t0] & ~kRaw, b1 = zt_off[t1] & ~kRaw;
      if (b1 > b0)
        SAI_CUDA_CHECK(cudaMemcpyAsync(static_cast<char*>(e->zt.p) + b0, zt_stream + b0, b1 - b0,
                                       cudaMemcpyHostToDevice, e->s_copy));
    }
    SAI_CUDA_CHECK(cudaEventRecord(e->ev[s], e->s_copy));
    SAI_CUDA_CHECK(cudaStreamWaitEvent(e->s_comp, e->ev[s], 0));
    if (zt)
      if (int rc = sai_zt_decode(lay, e->zt.p, zt_bytes, static_cast<const uint64_t*>(e->ztoff.p), t0, t1 - t0,
                                 e->packed.p, e->s_comp))
        return rc;
    if (int rc = sai_site_flags(lay, e->packed.p, t0, t1 - t0, n_tiles, jobs, n_jobs, d_mask_u,
                                d_mask_q, d_qval, stride, nullptr, nullptr, 0, 0, e->s_comp))
      return rc;
  }
  SAI_CUDA_CHECK(cudaEventRecord(e->ev[n_slices], e->s_copy));
  SAI_CUDA_CHECK(cudaStreamWaitEvent(e->s_comp, e->ev[n_slices], 0));
  return run_windows(e, out);
}

int sai_engine_score_host(sai_engine* e, const sai_layout* lay, const uint8_t* packed,
                          const int32_t* pos, int64_t n_sites, const int64_t* win_start,
                          const int64_t* win_end, int64_t n_windows, const sai_job* jobs,
                          int32_t n_jobs, sai_host_results* out) {
  SAI_REQUIRE(n_sites <= 0 || packed, "NULL input");
  return score_host_impl(e, lay, packed, nullptr, nullptr, nullptr, pos, n_sites, win_start, win_end, n_windows, jobs,
                         n_jobs, out);
}

int sai_engine_score_host_zt(sai_engine* e, const sai_layout* lay, const uint8_t* zt_stream,
                             const uint64_t* zt_tile_off, const int32_t* pos, int64_t n_sites,
                             const int64_t* win_start, const int64_t* win_end, int64_t n_windows,
                             const sai_job* jobs, int32_t n_jobs, sai_host_results* out) {
  SAI_REQUIRE(n_sites <= 0 || (zt_stream && zt_tile_off), "NULL input");
  return score_host_impl(e, lay, nullptr, zt_stream, zt_tile_off, nullptr, pos, n_sites, win_start, win_end, n_windows,
                         jobs, n_jobs, out);
}

int sai_engine_score_host_i8(sai_engine* e, const sai_layout* lay, const int8_t* const* gt,
                             const int64_t* row_stride, const int32_t* pos, int64_t n_sites,
                             const int64_t* win_start, const int64_t* win_end, int64_t n_windows,
                             const sai_job* jobs, int32_t n_jobs, sai_host_results* out) {
  SAI_REQUIRE(lay && gt && row_stride, "NULL input");
  if (int rc = validate_layout(lay)) return rc;
  for (int p = 0; p < lay->n_pops; ++p) {
    SAI_REQUIRE(n_sites <= 0 || gt[p], "NULL genotype matrix of population %d", p);
    SAI_REQUIRE(row_stride[p] >= lay->pop[p].n_samples, "row_stride of population %d smaller than n_samples", p);
  }
  const I8Source src{gt, row_stride};
  return score_host_impl(e, lay, nullptr, nullptr, nullptr, &src, pos, n_sites, win_start, win_end, n_windows, jobs,
                         n_jobs, out);
}

int sai_engine_set_i8_wire(sai_engine* e, int32_t mode) {
  SAI_REQUIRE(e, "NULL engine");
  SAI_REQUIRE(mode >= 0 && mode <= 2, "wire format: 0 = auto, 1 = dense tiles, 2 = zt records");
  e->i8_wire = mode;
  return SAI_OK;
}

uint64_t sai_engine_i8_wire_bytes(const sai_engine* e) { return e ? e->i8_wire_bytes : 0; }

int sai_engine_set_host_threads(sai_engine* e, int32_t n_threads) {
  SAI_REQUIRE(e, "NULL engine");
  e->host_threads = n_threads > 0 ? n_threads : 0;
  return SAI_OK;
}

int sai_engine_pattern_sums(sai_engine* e, const sai_layout* lay, int32_t ref_pop, int32_t tgt_pop,
                            int32_t out_pop, const int32_t* src_pops, int32_t n_src, double* sums) {
  SAI_REQUIRE(e && e->n_jobs > 0, "no previous sai_engine_score_host call");
  SAI_REQUIRE(sums && src_pops, "NULL argument");
  if (int rc = validate_layout(lay)) return rc;
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  const int64_t n_tiles = sai_num_tiles(e->n_sites);
  const int64_t stride = n_tiles * kTile;
  const int64_t W = e->W;
  if (W == 0 || n_src <= 0) return SAI_OK;
  if (int rc = grow(e->counts, sizeof(int32_t) * 2 * (size_t)lay->n_pops * stride + 256)) return rc;
  if (int rc = grow(e->sums, sizeof(double) * 7 * (size_t)n_src * W + 256)) return rc;
  int32_t* d_num = static_cast<int32_t*>(e->counts.p);
  int32_t* d_called = d_num + (size_t)lay->n_pops * stride;
  if (int rc = sai_site_counts(lay, e->packed.p, 0, n_tiles, d_num, d_called, stride, 0, e->s_comp)) return rc;
  const int64_t* d_ws = static_cast<const int64_t*>(e->win.p);
  const int32_t* d_pos = static_cast<const int32_t*>(e->pos.p);
  double* d_sums = static_cast<double*>(e->sums.p);
  // one sai_window_patterns per piece on its sites and counts; sums[k][w0 + i] <- piece's [k][i]
  for (const auto& P : scored_pieces(e)) {
    const int64_t w0 = P[0], nw = P[1], lo = P[2];
    if (nw == 0) continue;
    double* d_p = d_sums + 7 * (size_t)n_src * w0;
    if (int rc = sai_window_patterns(lay, d_pos + lo, P[3], d_ws + w0, d_ws + W + w0, nw, d_num + lo, d_called + lo,
                                     stride, ref_pop, tgt_pop, out_pop, src_pops, n_src, d_p, e->s_comp))
      return rc;
    SAI_CUDA_CHECK(cudaMemcpy2DAsync(sums + 7 * w0, sizeof(double) * 7 * W, d_p, sizeof(double) * 7 * nw,
                                     sizeof(double) * 7 * nw, n_src, cudaMemcpyDeviceToHost, e->s_comp));
  }
  SAI_CUDA_CHECK(cudaStreamSynchronize(e->s_comp));
  return SAI_OK;
}

// DD sums of both entry points over the pieces of the resident tiles.  P[j] = (first window, windows,
// first site, sites, row): the piece's entries of the negative-value table (d_ns / d_ni / d_nv, device)
// are those of offsets row `row` of neg_off ([rows][n_pops + 1], host), their sites counted from the
// piece's first site; row -1: a piece without sites, which has no entries.
static int dd_sums_impl(sai_engine* e, const sai_layout* lay, int32_t ref_pop, int32_t tgt_pop, const int32_t* src_pops,
                        int32_t n_src, int32_t m_max, const int32_t* d_ns, const int32_t* d_ni, const int32_t* d_nv,
                        const int64_t* neg_off, const std::vector<std::array<int64_t, 5>>& P, int64_t* ref_sum,
                        int64_t* tgt_sum) {
  const int n_pops = lay->n_pops;
  SAI_REQUIRE(ref_pop >= 0 && ref_pop < n_pops && tgt_pop >= 0 && tgt_pop < n_pops, "bad population index");
  SAI_REQUIRE(m_max >= 1, "m_max must be positive");
  SAI_REQUIRE(n_src <= SAI_MAX_SRC, "n_src %d outside [1,%d]", n_src, SAI_MAX_SRC);
  const int64_t W = e->W;
  if (W == 0 || n_src <= 0) return SAI_OK;
  // histograms of ref and tgt (what the distance kernels read) and, behind them, of the source
  // populations: only their missing-call totals are used, to check the table against the tiles
  int32_t hp[2 + SAI_MAX_SRC] = {ref_pop, tgt_pop};
  for (int k = 0; k < n_src; ++k) {
    SAI_REQUIRE(src_pops[k] >= 0 && src_pops[k] < n_pops, "bad source population index");
    hp[2 + k] = src_pops[k];
  }
  const int n_hp = 2 + n_src;
  int64_t max_stride = kTile;
  for (const auto& q : P) max_stride = std::max(max_stride, sai_num_tiles(q[3]) * kTile);
  const int64_t rows = sai_hist_rows(lay, hp, n_hp);
  const size_t out_n = (size_t)n_src * W * m_max;
  // [hist rows][uint64 missing totals per piece][int32 err] share the hist buffer
  const size_t hist_bytes = align256(sizeof(int32_t) * (size_t)rows * max_stride);
  if (int rc = grow(e->hist, hist_bytes + sizeof(uint64_t) * n_hp * P.size() + 256)) return rc;
  if (int rc = grow(e->dd, sizeof(int64_t) * 2 * out_n + 512)) return rc;
  cudaStream_t st = e->s_comp;
  int32_t* d_hist = static_cast<int32_t*>(e->hist.p);
  uint64_t* d_missing = reinterpret_cast<uint64_t*>(static_cast<char*>(e->hist.p) + hist_bytes);
  int32_t* d_err = reinterpret_cast<int32_t*>(d_missing + n_hp * P.size());
  int64_t* d_r = static_cast<int64_t*>(e->dd.p);
  int64_t* d_t = d_r + out_n;
  // a piece without sites leaves its missing totals untouched (sai_site_hist returns early): zero all of them
  SAI_CUDA_CHECK(cudaMemsetAsync(d_missing, 0, sizeof(uint64_t) * n_hp * P.size() + sizeof(int32_t), st));
  SAI_CUDA_CHECK(cudaMemsetAsync(d_r, 0, sizeof(int64_t) * 2 * out_n, st));
  const int64_t* d_ws = static_cast<const int64_t*>(e->win.p);
  const int32_t* d_pos = static_cast<const int32_t*>(e->pos.p);
  std::vector<int64_t> off((size_t)n_pops + 1);
  for (size_t j = 0; j < P.size(); ++j) {
    const int64_t w0 = P[j][0], nw = P[j][1], lo = P[j][2], n = P[j][3], c = P[j][4];
    if (nw == 0) continue;
    const int64_t base = c >= 0 ? neg_off[(size_t)c * (n_pops + 1)] : 0;
    for (int p = 0; p <= n_pops; ++p) off[p] = c >= 0 ? neg_off[(size_t)c * (n_pops + 1) + p] - base : 0;
    const void* packed = static_cast<const char*>(e->packed.p) + (size_t)(lo / kTile) * lay->pairs_per_site * kTile * 8;
    const int64_t stride = sai_num_tiles(n) * kTile;
    if (int rc = sai_site_hist(lay, packed, n, hp, n_hp, d_hist, stride, d_missing + n_hp * j, st)) return rc;
    int64_t* r = d_r + (size_t)n_src * m_max * w0;
    int64_t* t = d_t + (size_t)n_src * m_max * w0;
    if (int rc = sai_window_dd(lay, packed, d_pos + lo, n, d_ws + w0, d_ws + W + w0, nw, d_hist, stride, ref_pop, tgt_pop,
                               src_pops, n_src, off.data(), d_ns + base, d_ni + base, d_nv + base, r, t, m_max, d_err, st))
      return rc;
    const size_t row = sizeof(int64_t) * (size_t)nw * m_max, pitch = sizeof(int64_t) * (size_t)W * m_max;
    SAI_CUDA_CHECK(cudaMemcpy2DAsync(ref_sum + w0 * m_max, pitch, r, row, row, n_src, cudaMemcpyDeviceToHost, st));
    SAI_CUDA_CHECK(cudaMemcpy2DAsync(tgt_sum + w0 * m_max, pitch, t, row, row, n_src, cudaMemcpyDeviceToHost, st));
  }
  std::vector<uint64_t> h_missing((size_t)n_hp * P.size());
  int32_t h_err = 0;
  SAI_CUDA_CHECK(cudaMemcpyAsync(h_missing.data(), d_missing, sizeof(uint64_t) * h_missing.size(), cudaMemcpyDeviceToHost, st));
  SAI_CUDA_CHECK(cudaMemcpyAsync(&h_err, d_err, sizeof(h_err), cudaMemcpyDeviceToHost, st));
  SAI_CUDA_CHECK(cudaStreamSynchronize(st));
  // the bit-planes keep one missing code: every missing call needs its raw value in the table
  for (size_t j = 0; j < P.size(); ++j) {
    const int64_t c = P[j][4];
    if (P[j][1] == 0) continue;
    for (int q = 0; q < n_hp; ++q) {
      const size_t o = (size_t)c * (n_pops + 1) + hp[q];
      const int64_t have = c >= 0 ? neg_off[o + 1] - neg_off[o] : 0;
      SAI_REQUIRE((int64_t)h_missing[n_hp * j + q] == have,
                  "population %d has %lld missing calls but %lld entries in the negative-value table", hp[q],
                  (long long)h_missing[n_hp * j + q], (long long)have);
    }
  }
  SAI_REQUIRE(h_err == 0, "a missing source call has no entry in the negative-value table");
  return SAI_OK;
}

int sai_engine_dd_sums(sai_engine* e, const sai_layout* lay, int32_t ref_pop, int32_t tgt_pop,
                       const int32_t* src_pops, int32_t n_src, const int64_t* neg_off,
                       const int32_t* neg_site, const int32_t* neg_ind, const int32_t* neg_val,
                       int64_t* ref_sum, int64_t* tgt_sum, int32_t m_max) {
  SAI_REQUIRE(e && e->n_jobs > 0, "no previous sai_engine_score_host call");
  SAI_REQUIRE(ref_sum && tgt_sum && src_pops && neg_off, "NULL argument");
  if (int rc = validate_layout(lay)) return rc;
  SAI_REQUIRE(e->pieces.empty(), "sai_engine_dd_sums: the resident tiles are scored in pieces");
  const int64_t n_neg = neg_off[lay->n_pops];
  SAI_REQUIRE(n_neg >= 0 && (n_neg == 0 || (neg_site && neg_ind && neg_val)), "bad negative-value table");
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  if (int rc = grow(e->neg, sizeof(int32_t) * 3 * (size_t)n_neg + 256)) return rc;
  int32_t* d_ns = static_cast<int32_t*>(e->neg.p);
  int32_t* d_ni = d_ns + n_neg;
  int32_t* d_nv = d_ni + n_neg;
  if (n_neg > 0) {
    SAI_CUDA_CHECK(cudaMemcpyAsync(d_ns, neg_site, sizeof(int32_t) * n_neg, cudaMemcpyHostToDevice, e->s_comp));
    SAI_CUDA_CHECK(cudaMemcpyAsync(d_ni, neg_ind, sizeof(int32_t) * n_neg, cudaMemcpyHostToDevice, e->s_comp));
    SAI_CUDA_CHECK(cudaMemcpyAsync(d_nv, neg_val, sizeof(int32_t) * n_neg, cudaMemcpyHostToDevice, e->s_comp));
  }
  const auto q = scored_pieces(e)[0];  // the chunk is one piece, its entries the table's only row
  return dd_sums_impl(e, lay, ref_pop, tgt_pop, src_pops, n_src, m_max, d_ns, d_ni, d_nv, neg_off,
                      {{q[0], q[1], q[2], q[3], 0}}, ref_sum, tgt_sum);
}

int sai_engine_score_resident(sai_engine* e, const sai_job* jobs, int32_t n_jobs, sai_host_results* out) {
  SAI_REQUIRE(e && e->n_jobs > 0, "no previous sai_engine_score_host call");
  const sai_layout* lay = &e->lay;
  if (int rc = validate_jobs(lay, jobs, n_jobs)) return rc;
  if (int rc = check_results(out)) return rc;
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  const int64_t n_tiles = sai_num_tiles(e->n_sites);
  const int64_t stride = n_tiles * kTile;
  const ResLayout rl = res_layout(e->W, n_jobs);
  if (int rc = grow(e->mask, sizeof(uint32_t) * 2 * (size_t)n_jobs * n_tiles + 256)) return rc;
  if (int rc = grow(e->qval, sizeof(double) * (size_t)n_jobs * stride + 256)) return rc;
  if (int rc = grow(e->res, rl.total + 256)) return rc;
  e->n_jobs = n_jobs;
  for (int j = 0; j < n_jobs; ++j) e->jobs[j] = jobs[j];
  uint32_t* d_mask_u = static_cast<uint32_t*>(e->mask.p);
  if (n_tiles > 0)
    if (int rc = sai_site_flags(lay, e->packed.p, 0, n_tiles, n_tiles, jobs, n_jobs, d_mask_u,
                                d_mask_u + (size_t)n_jobs * n_tiles, static_cast<double*>(e->qval.p), stride, nullptr,
                                nullptr, 0, 0, e->s_comp))
      return rc;
  return run_windows(e, out);
}

int sai_engine_rescore_windows(sai_engine* e, sai_host_results* out) {
  SAI_REQUIRE(e && e->n_jobs > 0, "no previous sai_engine_score_host call");
  if (int rc = check_results(out)) return rc;
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  return run_windows(e, out);
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
// Ingest session (sai_engine_vcf_*): VCF text -> pinned ring slot (host threads) -> cudaMemcpyAsync on
// the copy stream -> sai_vcf_tiles_device on the compute stream, straight into the engine's tile and
// position buffers.  A host slot is rewritten once its copy has landed (`copied`), a device slot once
// the slice in it has been parsed (`parsed`).
namespace sai {

// vgen (genome ingest): hash table | name_off | anc_off | state | chroms | names, 256-byte aligned parts
struct GenLayout {
  size_t hash, name_off, anc_off, state, chroms, names, total;
};
static GenLayout gen_layout(int n_chrom, size_t name_bytes) {
  GenLayout g{};
  size_t at = 0;
  g.hash = at, at += align256(sizeof(uint32_t) * 2 * kChromHashSlots);
  g.name_off = at, at += align256(sizeof(int32_t) * (n_chrom + 1));
  g.anc_off = at, at += align256(sizeof(int64_t) * (n_chrom + 1));
  g.state = at, at += align256(sizeof(VcfGenomeState));
  g.chroms = at, at += align256(sizeof(VcfChromDev) * n_chrom);
  g.names = at, at += align256(name_bytes);
  g.total = at;
  return g;
}
static VcfGenomeState* vcf_genome_state(sai_engine* e) {
  return reinterpret_cast<VcfGenomeState*>(static_cast<char*>(e->vgen.p) + gen_layout(e->vcf.gq.n_chrom, 0).state);
}
static VcfChromDev* vcf_genome_chroms(sai_engine* e) {
  return reinterpret_cast<VcfChromDev*>(static_cast<char*>(e->vgen.p) + gen_layout(e->vcf.gq.n_chrom, 0).chroms);
}

// tile / position buffers for `cap` sites; `keep`: the sites parsed so far move along
static int vcf_grow_sites(sai_engine* e, int64_t cap, bool keep) {
  auto& V = e->vcf;
  cap = (cap + kTile - 1) / kTile * kTile;
  if (cap <= V.site_cap) return SAI_OK;
  const size_t tb = sai_packed_bytes(&V.q.lay, cap), pb = sizeof(int32_t) * (size_t)cap;
  if (keep) SAI_CUDA_CHECK(cudaStreamSynchronize(e->s_comp));
  const size_t old_tb = sai_packed_bytes(&V.q.lay, V.site_cap), old_pb = sizeof(int32_t) * (size_t)V.site_cap;
  for (auto [b, bytes, old] : {std::make_tuple(&e->packed, tb, old_tb), std::make_tuple(&e->pos, pb, old_pb)}) {
    if (bytes + 256 <= b->cap) continue;
    void* p = nullptr;
    cudaError_t ce = cudaMalloc(&p, bytes + 256);
    if (ce != cudaSuccess) {
      set_error("cudaMalloc(%zu) failed: %s", bytes + 256, cudaGetErrorString(ce));
      return SAI_E_NOMEM;
    }
    if (keep && old > 0 && b->p) SAI_CUDA_CHECK(cudaMemcpyAsync(p, b->p, old, cudaMemcpyDeviceToDevice, e->s_comp));
    if (keep) SAI_CUDA_CHECK(cudaStreamSynchronize(e->s_comp));
    if (b->p) SAI_CUDA_CHECK(cudaFree(b->p));
    b->p = p;
    b->cap = bytes + 256;
  }
  V.site_cap = cap;
  return SAI_OK;
}

// waits until `ev` has completed; any other answer than "not ready" is fatal
static int vcf_wait(cudaEvent_t ev) {
  for (;;) {
    const cudaError_t r = cudaEventQuery(ev);
    if (r == cudaSuccess) return SAI_OK;
    if (r != cudaErrorNotReady) {
      set_error("ingest ring: cudaEventQuery failed: %s", cudaGetErrorString(r));
      return SAI_E_CUDA;
    }
    std::this_thread::sleep_for(std::chrono::microseconds(20));
  }
}

// parse scratch of one slice of `len` bytes for the session's query
static uint64_t vcf_scratch_need(const sai_engine* e, int64_t len) {
  return (e->vcf.genome ? vcf_genome_scratch_bytes(e->vcf.gq, len) : sai_vcf_scratch_bytes(&e->vcf.q, len)) +
         (e->vcf.neg ? vcf_neg_scratch_bytes(e->vcf.q, len) : 0);
}

// The negative-value table of a session with n_chrom chromosomes (sai_engine_set_vcf_neg_table): its
// capacity is unknown until the text has been read.  First estimate: 1/64 of the site capacity times the
// individuals (about 1.6 % missing calls; the site capacity comes from the text size), at least 1024 and
// at least neg_min; finish reports SAI_E_CAPACITY and the true count when the text holds more, and the
// caller reads the text again.
constexpr int64_t kNegMaxEntries = (int64_t(1) << 31) - 1;  // site / individual / index are int32
static int vcf_neg_begin(sai_engine* e, int32_t n_chrom) {
  auto& V = e->vcf;
  V.neg = V.neg_on;
  V.neg_n = -1;
  V.neg_off.clear();
  V.chrom_sites.clear();
  if (!V.neg) return SAI_OK;
  const sai_layout& lay = V.q.lay;
  int64_t n_out = 0;
  for (int p = 0; p < lay.n_pops; ++p) n_out += lay.pop[p].n_samples;
  const int64_t cap = std::min(kNegMaxEntries, std::max(V.neg_min, std::max<int64_t>(1024, V.site_cap / 64 * n_out)));
  const size_t part = align256(sizeof(int32_t) * (size_t)cap);
  if (int rc = grow(e->vnega, 5 * part)) return rc;
  const size_t count_bytes = sizeof(unsigned long long) * (size_t)n_chrom * lay.n_pops;
  if (int rc = grow(e->vneg, align256(sizeof(VcfNegDev)) + count_bytes)) return rc;
  VcfNegSession& t = V.negs;
  char* a = static_cast<char*>(e->vnega.p);
  t.site = reinterpret_cast<int32_t*>(a);
  t.ind = reinterpret_cast<int32_t*>(a + part);
  t.val = reinterpret_cast<int32_t*>(a + 2 * part);
  t.key = reinterpret_cast<int32_t*>(a + 3 * part);
  t.idx = reinterpret_cast<int32_t*>(a + 4 * part);
  t.cap = cap;
  t.state = static_cast<VcfNegDev*>(e->vneg.p);
  t.count = reinterpret_cast<unsigned long long*>(static_cast<char*>(e->vneg.p) + align256(sizeof(VcfNegDev)));
  SAI_CUDA_CHECK(cudaMemsetAsync(e->vneg.p, 0, align256(sizeof(VcfNegDev)) + count_bytes, e->s_comp));
  return SAI_OK;
}

// After a successful finish: the appended entries placed key-major (chromosome, population; inside a
// key by site and individual) into vnegt, and their offsets.
static int vcf_neg_finish(sai_engine* e) {
  auto& V = e->vcf;
  const int n_chrom = V.genome ? V.gq.n_chrom : 1, n_pops = V.q.lay.n_pops;
  const int64_t n = V.neg_n;
  std::vector<unsigned long long> count((size_t)n_chrom * n_pops);
  SAI_CUDA_CHECK(cudaMemcpy(count.data(), V.negs.count, sizeof(unsigned long long) * count.size(), cudaMemcpyDeviceToHost));
  std::vector<int64_t> key_off(count.size() + 1, 0);
  for (size_t k = 0; k < count.size(); ++k) key_off[k + 1] = key_off[k] + (int64_t)count[k];
  SAI_REQUIRE(key_off.back() == n, "negative-value table: %lld entries appended, %lld counted", (long long)n,
              (long long)key_off.back());
  V.neg_off.assign((size_t)n_chrom * (n_pops + 1), 0);
  for (int c = 0; c < n_chrom; ++c)
    for (int p = 0; p <= n_pops; ++p) V.neg_off[(size_t)c * (n_pops + 1) + p] = key_off[(size_t)c * n_pops + p];
  const size_t part = align256(sizeof(int32_t) * (size_t)std::max<int64_t>(n, 1));
  if (int rc = grow(e->vnegt, 3 * part + sizeof(int64_t) * key_off.size())) return rc;
  char* t = static_cast<char*>(e->vnegt.p);
  int64_t* d_key_off = reinterpret_cast<int64_t*>(t + 3 * part);
  SAI_CUDA_CHECK(cudaMemcpyAsync(d_key_off, key_off.data(), sizeof(int64_t) * key_off.size(), cudaMemcpyHostToDevice, e->s_comp));
  if (int rc = vcf_neg_order(V.negs, n, d_key_off, reinterpret_cast<int32_t*>(t), reinterpret_cast<int32_t*>(t + part),
                             reinterpret_cast<int32_t*>(t + 2 * part), e->s_comp))
    return rc;
  SAI_CUDA_CHECK(cudaStreamSynchronize(e->s_comp));  // key_off goes out of scope
  return SAI_OK;
}

static int stage_threads(const sai_engine* e) {
  return std::min(16, e->host_threads > 0 ? e->host_threads : (int)std::max(1u, std::thread::hardware_concurrency()));
}

static double now_s() {
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// The host slot of the next slice, with room for `n` bytes (the ring grows -- after a drain -- when a
// slice is larger than its slots) and free: the H2D copy of the slice that used it last has landed.
static int vcf_acquire_slot(sai_engine* e, int64_t n, char** h) {
  auto& V = e->vcf;
  if ((size_t)n + 16 > V.slot_bytes) {
    SAI_CUDA_CHECK(cudaStreamSynchronize(e->s_copy));
    SAI_CUDA_CHECK(cudaStreamSynchronize(e->s_comp));
    const size_t want = std::max<size_t>((size_t)n + 16, std::min<size_t>((size_t)V.slice_bytes + 16, 2 * V.slot_bytes + (1u << 20)));
    const size_t slot = align256(want);
    if (V.h_ring) SAI_CUDA_CHECK(cudaFreeHost(V.h_ring));
    V.h_ring = nullptr;
    V.slot_bytes = 0;
    SAI_CUDA_CHECK(cudaHostAlloc(reinterpret_cast<void**>(&V.h_ring), slot * V.ring, cudaHostAllocDefault));
    if (int rc = grow(e->vtext, slot * V.ring)) return rc;
    if (int rc = grow(e->vscratch, vcf_scratch_need(e, (int64_t)slot))) return rc;
    V.slot_bytes = slot;
  }
  while ((int)V.copied.size() < V.ring) {
    cudaEvent_t a, b;
    SAI_CUDA_CHECK(cudaEventCreateWithFlags(&a, cudaEventDisableTiming));
    SAI_CUDA_CHECK(cudaEventCreateWithFlags(&b, cudaEventDisableTiming));
    V.copied.push_back(a);
    V.parsed.push_back(b);
  }
  const int slot = (int)(V.n_slices % V.ring);
  if (V.n_slices >= V.ring) {
    const double t0 = now_s();
    const int rc = vcf_wait(V.copied[slot]);
    V.t_wait += now_s() - t0;
    if (rc) return rc;
  }
  *h = V.h_ring + (size_t)slot * V.slot_bytes;
  return SAI_OK;
}

// A compressed group in the slot's part of the compressed ring (device inflate): `bytes` to copy,
// starting with `n_desc` block descriptors; descriptor i is block first_block + i (the carry's
// pseudo-blocks come last).
struct DevGroup {
  size_t bytes;
  int64_t n_desc, first_block;
};

// Bytes [off, off + n) of the acquired slot (complete lines) -> device slot (copy stream) -> parse (compute stream).
// With `g` the slot's compressed group goes over instead and is inflated into the device slot on the slot's
// own inflate stream: one slice has too few blocks to fill the GPU, so the inflates of the slices in the
// ring run side by side (and next to the parse); [off, off + n) is then the range of the inflated text
// that is parsed.  The slot's inflate waits for its copy, which waited for the slot's previous parse.
static int vcf_launch_slot_impl(sai_engine* e, int64_t off, int64_t n, const DevGroup* g);
static int vcf_launch_slot(sai_engine* e, int64_t off, int64_t n, const DevGroup* g = nullptr) {
  const double t0 = now_s();
  const int rc = vcf_launch_slot_impl(e, off, n, g);
  e->vcf.t_launch += now_s() - t0;
  return rc;
}
static int vcf_launch_slot_impl(sai_engine* e, int64_t off, int64_t n, const DevGroup* g) {
  auto& V = e->vcf;
  V.fed += n;
  // records of normal width in the text so far (+ a tile of padding per chromosome of a genome parse)
  const int64_t need = V.fed / V.row_bytes + V.n_slices + 1 + 1024 + (V.genome ? (int64_t)kTile * V.gq.n_chrom : 0);
  if (need > V.site_cap)
    if (int rc = vcf_grow_sites(e, std::max(need, 2 * V.site_cap), true)) return rc;
  while ((int64_t)V.tev.size() <= V.n_slices) {
    std::array<cudaEvent_t, 6> t;
    for (auto& x : t) SAI_CUDA_CHECK(cudaEventCreate(&x));
    V.tev.push_back(t);
  }
  V.inflated.resize((size_t)V.n_slices + 1);
  V.inflated[V.n_slices] = g != nullptr;
  const auto& T = V.tev[V.n_slices];
  const int slot = (int)(V.n_slices % V.ring);
  char* d = static_cast<char*>(e->vtext.p) + (size_t)slot * V.slot_bytes;
  if (V.n_slices >= V.ring) SAI_CUDA_CHECK(cudaStreamWaitEvent(e->s_copy, V.parsed[slot], 0));
  SAI_CUDA_CHECK(cudaEventRecord(T[0], e->s_copy));
  if (!g) {
    SAI_CUDA_CHECK(cudaMemcpyAsync(d, V.h_ring + (size_t)slot * V.slot_bytes + off, (size_t)n, cudaMemcpyHostToDevice,
                                   e->s_copy));
  } else {
    uint8_t* dc = static_cast<uint8_t*>(e->vcomp.p) + (size_t)slot * V.comp_slot;
    SAI_CUDA_CHECK(cudaMemcpyAsync(dc, V.h_comp + (size_t)slot * V.comp_slot, g->bytes, cudaMemcpyHostToDevice, e->s_copy));
    V.comp_bytes += (double)g->bytes;
  }
  SAI_CUDA_CHECK(cudaEventRecord(T[1], e->s_copy));
  SAI_CUDA_CHECK(cudaEventRecord(V.copied[slot], e->s_copy));
  if (g) {
    uint8_t* dc = static_cast<uint8_t*>(e->vcomp.p) + (size_t)slot * V.comp_slot;
    int32_t* status = reinterpret_cast<int32_t*>(dc + align256(g->bytes));
    while ((int)V.s_infl.size() <= slot) {
      cudaStream_t s;
      SAI_CUDA_CHECK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
      V.s_infl.push_back(s);
    }
    cudaStream_t si = V.s_infl[slot];
    SAI_CUDA_CHECK(cudaStreamWaitEvent(si, V.copied[slot], 0));
    SAI_CUDA_CHECK(cudaEventRecord(T[4], si));
    if (int rc = bgzf_inflate_launch(dc, reinterpret_cast<const sai_bgzf_block*>(dc), g->n_desc, reinterpret_cast<uint8_t*>(d),
                                     status, static_cast<unsigned long long*>(e->vbad.p), g->first_block, si))
      return rc;
    SAI_CUDA_CHECK(cudaEventRecord(T[5], si));
    SAI_CUDA_CHECK(cudaStreamWaitEvent(e->s_comp, T[5], 0));
    d += off;
  } else {
    SAI_CUDA_CHECK(cudaStreamWaitEvent(e->s_comp, V.copied[slot], 0));
  }
  SAI_CUDA_CHECK(cudaEventRecord(T[2], e->s_comp));
  const VcfNegSession* neg = V.neg ? &V.negs : nullptr;
  if (int rc = V.genome ? vcf_tiles_genome(V.gq, d, n, e->vscratch.p, e->vscratch.cap, e->packed.p,
                                            static_cast<int32_t*>(e->pos.p), V.site_cap,
                                            static_cast<sai_vcf_state*>(e->vstate.p), vcf_genome_state(e),
                                            vcf_genome_chroms(e), neg, e->s_comp)
                       : vcf_tiles_single(V.q, d, n, e->vscratch.p, e->vscratch.cap, e->packed.p,
                                          static_cast<int32_t*>(e->pos.p), V.site_cap,
                                          static_cast<sai_vcf_state*>(e->vstate.p), neg, e->s_comp))
    return rc;
  SAI_CUDA_CHECK(cudaEventRecord(T[3], e->s_comp));
  SAI_CUDA_CHECK(cudaEventRecord(V.parsed[slot], e->s_comp));
  ++V.n_slices;
  return SAI_OK;
}

// host text -> pinned slot, 1 MB parts over the staging threads
static void staged_copy(sai_engine* e, char* dst, const char* src, size_t n) {
  const size_t part = 1u << 20;
  const double t0 = now_s();
  const std::function<void(int64_t)> f = [&](int64_t i) {
    const size_t a = (size_t)i * part;
    memcpy(dst + a, src + a, std::min(part, n - a));
  };
  e->vcf.pool.run(stage_threads(e), (int64_t)((n + part - 1) / part), f);
  e->vcf.t_stage += now_s() - t0;
}

}  // namespace sai

extern "C" {

int sai_engine_vcf_begin(sai_engine* e, const sai_layout* lay, const char* chrom, int64_t start, int64_t end,
                         const int32_t* sample_column, int32_t n_out, const int32_t* anc_pos,
                         const char* anc_allele, int64_t n_anc, int32_t n_file_samples, int64_t text_bytes_hint,
                         int64_t min_sites) {
  SAI_REQUIRE(e && lay && chrom && sample_column, "sai_engine_vcf_begin: NULL argument");
  if (int rc = validate_layout(lay)) return rc;
  int64_t total = 0;
  for (int p = 0; p < lay->n_pops; ++p) total += lay->pop[p].n_samples;
  SAI_REQUIRE(total == n_out, "sai_engine_vcf_begin: n_out %d != individuals of the layout %lld", n_out, (long long)total);
  const size_t clen = strlen(chrom);
  SAI_REQUIRE(clen >= 1 && clen < sizeof(sai_vcf_query::chrom), "sai_engine_vcf_begin: chromosome name of %zu bytes (1..255)", clen);
  SAI_REQUIRE(n_anc >= 0 && (n_anc == 0 || (anc_pos && anc_allele)), "sai_engine_vcf_begin: bad ancestral-allele table");
  SAI_REQUIRE(n_file_samples >= 0 && text_bytes_hint >= 0 && min_sites >= 0, "sai_engine_vcf_begin: negative size");
  int32_t max_col = 0;
  for (int i = 0; i < n_out; ++i) {
    SAI_REQUIRE(sample_column[i] >= 0, "sai_engine_vcf_begin: negative sample column");
    max_col = std::max(max_col, sample_column[i]);
  }
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  auto& V = e->vcf;
  if (V.state == 1) {  // an unfinished session: let its work drain before its buffers are reused
    SAI_CUDA_CHECK(cudaStreamSynchronize(e->s_copy));
    SAI_CUDA_CHECK(cudaStreamSynchronize(e->s_comp));
  }
  V.state = 0;
  V.genome = false;
  e->n_jobs = 0;  // the resident chunk is replaced
  e->pieces.clear();
  sai_vcf_query& q = V.q;
  q = sai_vcf_query{};
  q.lay = *lay;
  q.start = start;
  q.end = end;
  q.n_anc = n_anc;
  q.max_column = max_col;
  q.chrom_len = (int32_t)clen;
  memcpy(q.chrom, chrom, clen);
  if (int rc = grow(e->vcols, sizeof(int32_t) * (size_t)n_out)) return rc;
  SAI_CUDA_CHECK(cudaMemcpy(e->vcols.p, sample_column, sizeof(int32_t) * (size_t)n_out, cudaMemcpyHostToDevice));
  q.sample_column = static_cast<const int32_t*>(e->vcols.p);
  if (n_anc > 0) {
    if (int rc = grow(e->vanc_pos, sizeof(int32_t) * (size_t)n_anc)) return rc;
    if (int rc = grow(e->vanc_all, 8 * (size_t)n_anc)) return rc;
    SAI_CUDA_CHECK(cudaMemcpy(e->vanc_pos.p, anc_pos, sizeof(int32_t) * (size_t)n_anc, cudaMemcpyHostToDevice));
    SAI_CUDA_CHECK(cudaMemcpy(e->vanc_all.p, anc_allele, 8 * (size_t)n_anc, cudaMemcpyHostToDevice));
    q.anc_pos = static_cast<const int32_t*>(e->vanc_pos.p);
    q.anc_allele = static_cast<const char*>(e->vanc_all.p);
  }
  if (int rc = grow(e->vstate, sizeof(sai_vcf_state))) return rc;
  SAI_CUDA_CHECK(cudaMemsetAsync(e->vstate.p, 0, sizeof(sai_vcf_state), e->s_comp));
  V.row_bytes = std::max<int64_t>(64, 2 * (int64_t)n_file_samples + 18);
  V.site_cap = 0;  // the buffers' content is not kept from an earlier chunk
  if (int rc = vcf_grow_sites(e, std::max(text_bytes_hint / V.row_bytes + 1024, min_sites), false)) return rc;
  if (int rc = vcf_neg_begin(e, 1)) return rc;
  if (V.slot_bytes > 0)  // the scratch depends on the query (max_column): resize for the ring's slots
    if (int rc = grow(e->vscratch, vcf_scratch_need(e, (int64_t)V.slot_bytes))) return rc;
  if (int rc = grow(e->vbad, sizeof(unsigned long long))) return rc;
  SAI_CUDA_CHECK(cudaMemsetAsync(e->vbad.p, 0xff, sizeof(unsigned long long), e->s_copy));  // no corrupt block
  V.fed = V.n_slices = 0;
  V.t_stage = V.t_wait = V.t_launch = V.t_feed = V.t_boundary = V.comp_bytes = 0;
  V.carry.clear();
  V.sticky_rc = SAI_OK;
  V.state = 1;
  return SAI_OK;
}

static int vcf_feed_impl(sai_engine* e, const char* text, int64_t len, int64_t* consumed);
int sai_engine_vcf_feed(sai_engine* e, const char* text, int64_t len, int64_t* consumed) {
  const double t0 = now_s();
  const int rc = vcf_feed_impl(e, text, len, consumed);
  if (e) e->vcf.t_feed += now_s() - t0;
  return rc;
}
static int vcf_feed_impl(sai_engine* e, const char* text, int64_t len, int64_t* consumed) {
  SAI_REQUIRE(e && consumed && len >= 0 && (len == 0 || text), "sai_engine_vcf_feed: bad argument");
  *consumed = 0;
  auto& V = e->vcf;
  SAI_REQUIRE(V.state == 1, "sai_engine_vcf_feed: no ingest session (sai_engine_vcf_begin)");
  if (V.sticky_rc) return V.sticky_rc;
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  const void* last = len > 0 ? memrchr(text, '\n', (size_t)len) : nullptr;
  if (!last) return SAI_OK;
  const int64_t complete = static_cast<const char*>(last) - text + 1;
  int64_t at = 0;
  while (at < complete) {
    const int64_t want = std::min<int64_t>(complete - at, V.slice_bytes);
    int64_t cut = at + want;
    if (cut < complete) {  // end the slice after its last complete line; a longer line makes a longer slice
      const void* nl = memrchr(text + at, '\n', (size_t)want);
      if (!nl) nl = memchr(text + cut, '\n', (size_t)(complete - cut));
      cut = static_cast<const char*>(nl) - text + 1;
    }
    if (cut - at >= (int64_t(1) << 31)) {
      set_error("sai_engine_vcf_feed: a line of more than 2 GB");
      V.sticky_rc = SAI_E_ARG;
      return SAI_E_ARG;
    }
    char* h = nullptr;
    int rc = vcf_acquire_slot(e, cut - at, &h);
    if (rc == SAI_OK) {
      staged_copy(e, h, text + at, (size_t)(cut - at));
      rc = vcf_launch_slot(e, 0, cut - at);
    }
    if (rc) {
      V.sticky_rc = rc;
      return rc;
    }
    at = cut;
  }
  *consumed = complete;
  return SAI_OK;
}

static int vcf_finish_impl(sai_engine* e, int64_t* n_sites, int32_t* max_value, int32_t* pos_out, int64_t pos_cap);
int sai_engine_vcf_finish(sai_engine* e, int64_t* n_sites, int32_t* max_value, int32_t* pos_out, int64_t pos_cap) {
  SAI_REQUIRE(e && n_sites && max_value, "sai_engine_vcf_finish: NULL argument");
  SAI_REQUIRE(!e->vcf.genome, "sai_engine_vcf_finish: a genome session ends with sai_engine_vcf_genome_finish");
  return vcf_finish_impl(e, n_sites, max_value, pos_out, pos_cap);
}

int sai_engine_vcf_genome_begin(sai_engine* e, const sai_layout* lay, const char* names, const int32_t* name_off,
                                int32_t n_chrom, const int32_t* sample_column, int32_t n_out, const int32_t* anc_pos,
                                const char* anc_allele, const int64_t* anc_off, int32_t n_file_samples,
                                int64_t text_bytes_hint, int64_t min_sites) {
  SAI_REQUIRE(e && names && name_off, "sai_engine_vcf_genome_begin: NULL argument");
  std::vector<uint32_t> table(2 * kChromHashSlots);
  if (int rc = vcf_chrom_table(names, name_off, n_chrom, table.data())) return rc;
  const int64_t n_anc = anc_off ? anc_off[n_chrom] : 0;
  for (int c = 0; anc_off && c < n_chrom; ++c)
    SAI_REQUIRE(anc_off[0] == 0 && anc_off[c] <= anc_off[c + 1], "sai_engine_vcf_genome_begin: bad ancestral-table offsets");
  const std::string first(names + name_off[0], names + name_off[1]);
  if (int rc = sai_engine_vcf_begin(e, lay, first.c_str(), 1, 0, sample_column, n_out, anc_pos, anc_allele, n_anc,
                                    n_file_samples, text_bytes_hint, min_sites))
    return rc;
  auto& V = e->vcf;
  V.state = 0;  // until the table is in place
  const GenLayout gl = gen_layout(n_chrom, (size_t)name_off[n_chrom]);
  if (int rc = grow(e->vgen, gl.total)) return rc;
  char* g = static_cast<char*>(e->vgen.p);
  std::vector<int64_t> aoff(n_chrom + 1, 0);
  if (anc_off) std::copy(anc_off, anc_off + n_chrom + 1, aoff.begin());
  SAI_CUDA_CHECK(cudaMemcpyAsync(g + gl.hash, table.data(), sizeof(uint32_t) * table.size(), cudaMemcpyHostToDevice, e->s_comp));
  SAI_CUDA_CHECK(cudaMemcpyAsync(g + gl.name_off, name_off, sizeof(int32_t) * (n_chrom + 1), cudaMemcpyHostToDevice, e->s_comp));
  SAI_CUDA_CHECK(cudaMemcpyAsync(g + gl.anc_off, aoff.data(), sizeof(int64_t) * (n_chrom + 1), cudaMemcpyHostToDevice, e->s_comp));
  SAI_CUDA_CHECK(cudaMemcpyAsync(g + gl.names, names, (size_t)name_off[n_chrom], cudaMemcpyHostToDevice, e->s_comp));
  SAI_CUDA_CHECK(cudaStreamSynchronize(e->s_comp));  // the host vectors go out of scope
  VcfGenomeQuery& gq = V.gq;
  gq = VcfGenomeQuery{};
  gq.q = V.q;
  gq.anc_off = reinterpret_cast<const int64_t*>(g + gl.anc_off);
  gq.names = g + gl.names;
  gq.name_off = reinterpret_cast<const int32_t*>(g + gl.name_off);
  gq.hash = reinterpret_cast<const uint32_t*>(g + gl.hash);
  gq.n_chrom = n_chrom;
  V.genome = true;
  if (int rc = vcf_genome_state_init(vcf_genome_state(e), vcf_genome_chroms(e), n_chrom, e->s_comp)) return rc;
  if (int rc = vcf_grow_sites(e, V.site_cap + (int64_t)kTile * n_chrom, false)) return rc;
  if (int rc = vcf_neg_begin(e, n_chrom)) return rc;
  if (V.slot_bytes > 0)
    if (int rc = grow(e->vscratch, vcf_scratch_need(e, (int64_t)V.slot_bytes))) return rc;
  V.state = 1;
  return SAI_OK;
}

int sai_engine_vcf_genome_finish(sai_engine* e, int64_t* n_sites, int32_t* max_value, sai_vcf_chrom* chroms,
                                 int32_t* pos_out, int64_t pos_cap) {
  SAI_REQUIRE(e && n_sites && max_value && chroms, "sai_engine_vcf_genome_finish: NULL argument");
  auto& V = e->vcf;
  SAI_REQUIRE(V.genome, "sai_engine_vcf_genome_finish: no genome session (sai_engine_vcf_genome_begin)");
  const int rc = vcf_finish_impl(e, n_sites, max_value, pos_out, pos_cap);
  if (rc != SAI_OK && rc != SAI_E_CAPACITY && rc != SAI_E_DOMAIN) return rc;
  const int n = V.gq.n_chrom;
  VcfGenomeState gs;
  std::vector<VcfChromDev> dev(n);
  SAI_CUDA_CHECK(cudaMemcpy(&gs, vcf_genome_state(e), sizeof(gs), cudaMemcpyDeviceToHost));
  SAI_CUDA_CHECK(cudaMemcpy(dev.data(), vcf_genome_chroms(e), sizeof(VcfChromDev) * n, cudaMemcpyDeviceToHost));
  for (int c = 0; c < n; ++c) {
    const VcfChromDev& d = dev[c];
    const bool any = d.n_records > 0;
    chroms[c] = sai_vcf_chrom{any ? (int64_t)(uint32_t)d.first_key : 0, any ? (int64_t)(uint32_t)d.last_key : 0,
                              d.n_records, d.first_site, d.n_sites};
  }
  V.chrom_sites.resize((size_t)n);
  for (int c = 0; c < n; ++c) V.chrom_sites[c] = {dev[c].first_site, dev[c].n_sites};
  if (gs.noncontiguous) {
    V.state = 0;
    set_error("a chromosome's records resume after another chromosome's");
    return SAI_E_ORDER;
  }
  return rc;
}

static int vcf_finish_impl(sai_engine* e, int64_t* n_sites, int32_t* max_value, int32_t* pos_out, int64_t pos_cap) {
  auto& V = e->vcf;
  SAI_REQUIRE(V.state == 1, "sai_engine_vcf_finish: no ingest session (sai_engine_vcf_begin)");
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  V.state = 0;
  const double t_sync = now_s();
  const cudaError_t c1 = cudaStreamSynchronize(e->s_copy), c2 = cudaStreamSynchronize(e->s_comp);
  double h2d = 0, parse = 0, span = 0, infl = 0;
  int64_t n_inflated = 0;
  float ms = 0;
  for (int64_t k = 0; c1 == cudaSuccess && c2 == cudaSuccess && k < V.n_slices; ++k) {
    const auto& T = V.tev[k];
    if (cudaEventElapsedTime(&ms, T[0], T[1]) == cudaSuccess) h2d += ms / 1e3;
    if (cudaEventElapsedTime(&ms, T[2], T[3]) == cudaSuccess) parse += ms / 1e3;
    if (V.inflated[k]) {
      ++n_inflated;
      if (cudaEventElapsedTime(&ms, T[4], T[5]) == cudaSuccess) infl += ms / 1e3;
    }
  }
  if (c1 == cudaSuccess && c2 == cudaSuccess && V.n_slices > 0 &&
      cudaEventElapsedTime(&ms, V.tev[0][0], V.tev[V.n_slices - 1][3]) == cudaSuccess)
    span = ms / 1e3;
  const double stats[14] = {V.t_stage, V.t_wait, h2d, parse, span, (double)V.n_slices, (double)V.fed, now_s() - t_sync,
                            V.t_launch, V.t_feed, infl, V.comp_bytes, V.t_boundary, (double)n_inflated};
  memcpy(V.stats, stats, sizeof(stats));
  if (V.sticky_rc) {
    set_error("ingest session failed earlier (code %d)", V.sticky_rc);
    return V.sticky_rc;
  }
  if (c1 != cudaSuccess || c2 != cudaSuccess) {
    set_error("ingest session: %s", cudaGetErrorString(c1 != cudaSuccess ? c1 : c2));
    return SAI_E_CUDA;
  }
  if (n_inflated > 0) {
    unsigned long long bad = 0;
    SAI_CUDA_CHECK(cudaMemcpy(&bad, e->vbad.p, sizeof(bad), cudaMemcpyDeviceToHost));
    if (bad != ~0ull) {
      set_error("BGZF block %lld is corrupt", (long long)bad);
      return SAI_E_CORRUPT;
    }
  }
  sai_vcf_state st;
  SAI_CUDA_CHECK(cudaMemcpy(&st, e->vstate.p, sizeof(st), cudaMemcpyDeviceToHost));
  *n_sites = st.n_sites;
  const sai_layout& lay = V.q.lay;
  bool fits = true;
  for (int p = 0; p < lay.n_pops; ++p) {
    max_value[p] = std::max(lay.pop[p].ploidy, st.vmax[p]);
    if (max_value[p] > (1 << lay.pop[p].bits) - 2) fits = false;
  }
  if (V.neg) {
    VcfNegDev nd;
    SAI_CUDA_CHECK(cudaMemcpy(&nd, V.negs.state, sizeof(nd), cudaMemcpyDeviceToHost));
    V.neg_n = (int64_t)nd.n;
  }
  if (st.overflow) {
    set_error("more records than the ingest buffers hold (%lld sites, room for %lld)", (long long)st.n_sites,
              (long long)V.site_cap);
    return SAI_E_CAPACITY;
  }
  if (V.neg && V.neg_n > V.negs.cap) {
    set_error("more missing calls than the negative-value table holds (%lld entries, room for %lld)",
              (long long)V.neg_n, (long long)V.negs.cap);
    return SAI_E_CAPACITY;
  }
  if (!fits) {
    set_error("a genotype value does not fit the bit-planes of its population");
    return SAI_E_DOMAIN;
  }
  if (pos_out && pos_cap >= st.n_sites && st.n_sites > 0)
    SAI_CUDA_CHECK(cudaMemcpy(pos_out, e->pos.p, sizeof(int32_t) * (size_t)st.n_sites, cudaMemcpyDeviceToHost));
  if (V.neg)
    if (int rc = vcf_neg_finish(e)) return rc;
  e->n_sites = st.n_sites;
  e->lay = lay;
  e->n_jobs = 0;
  e->W = 0;
  V.state = 2;
  return SAI_OK;
}

static int score_loaded_impl(sai_engine* e, const int64_t* win_start, const int64_t* win_end, int64_t n_windows,
                             const sai_job* jobs, int32_t n_jobs, sai_host_results* out,
                             const std::vector<std::array<int64_t, 4>>& pieces);
int sai_engine_score_loaded(sai_engine* e, const int64_t* win_start, const int64_t* win_end, int64_t n_windows,
                            const sai_job* jobs, int32_t n_jobs, sai_host_results* out) {
  return score_loaded_impl(e, win_start, win_end, n_windows, jobs, n_jobs, out, {});
}

int sai_engine_score_loaded_pieces(sai_engine* e, const int64_t* win_start, const int64_t* win_end,
                                   const int64_t* pieces, int32_t n_pieces, const sai_job* jobs, int32_t n_jobs,
                                   sai_host_results* out) {
  SAI_REQUIRE(e && e->vcf.state == 2, "sai_engine_score_loaded_pieces: no finished ingest session");
  SAI_REQUIRE(n_pieces >= 1 && pieces, "sai_engine_score_loaded_pieces: no pieces");
  std::vector<std::array<int64_t, 4>> P((size_t)n_pieces);
  int64_t W = 0;
  for (int p = 0; p < n_pieces; ++p) {
    const int64_t nw = pieces[3 * p], lo = pieces[3 * p + 1], n = pieces[3 * p + 2];
    SAI_REQUIRE(nw >= 0 && lo >= 0 && lo % kTile == 0 && n >= 0 && lo + n <= e->n_sites,
                "sai_engine_score_loaded_pieces: piece %d (%lld windows, sites %lld + %lld) outside the %lld resident sites",
                p, (long long)nw, (long long)lo, (long long)n, (long long)e->n_sites);
    P[p] = {W, nw, lo, n};
    W += nw;
  }
  return score_loaded_impl(e, win_start, win_end, W, jobs, n_jobs, out, P);
}

static int score_loaded_impl(sai_engine* e, const int64_t* win_start, const int64_t* win_end, int64_t n_windows,
                             const sai_job* jobs, int32_t n_jobs, sai_host_results* out,
                             const std::vector<std::array<int64_t, 4>>& pieces) {
  SAI_REQUIRE(e && e->vcf.state == 2, "sai_engine_score_loaded: no finished ingest session");
  if (int rc = validate_jobs(&e->lay, jobs, n_jobs)) return rc;
  if (int rc = check_results(out)) return rc;
  SAI_REQUIRE(n_windows >= 0 && (n_windows == 0 || (win_start && win_end)), "NULL windows");
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  const int64_t W = n_windows;
  const int64_t n_tiles = sai_num_tiles(e->n_sites);
  const int64_t stride = n_tiles * kTile;
  const ResLayout rl = res_layout(W, n_jobs);
  // window bounds, then (pieces) each window's first and last site
  if (int rc = grow(e->win, (sizeof(int64_t) + sizeof(int32_t)) * 2 * (size_t)W + 256)) return rc;
  if (int rc = grow(e->mask, sizeof(uint32_t) * 2 * (size_t)n_jobs * n_tiles + 256)) return rc;
  if (int rc = grow(e->qval, sizeof(double) * (size_t)n_jobs * stride + 256)) return rc;
  if (int rc = grow(e->res, rl.total + 256)) return rc;
  e->W = W;
  e->n_jobs = n_jobs;
  e->pieces = pieces;
  for (int j = 0; j < n_jobs; ++j) e->jobs[j] = jobs[j];
  int64_t* d_ws = static_cast<int64_t*>(e->win.p);
  if (W > 0) {
    SAI_CUDA_CHECK(cudaMemcpyAsync(d_ws, win_start, sizeof(int64_t) * W, cudaMemcpyHostToDevice, e->s_comp));
    SAI_CUDA_CHECK(cudaMemcpyAsync(d_ws + W, win_end, sizeof(int64_t) * W, cudaMemcpyHostToDevice, e->s_comp));
  }
  if (!pieces.empty() && W > 0) {
    std::vector<int32_t> fl(2 * (size_t)W);
    for (const auto& P : pieces)
      for (int64_t i = P[0]; i < P[0] + P[1]; ++i) {
        fl[i] = (int32_t)P[2];
        fl[W + i] = (int32_t)(P[2] + P[3]);
      }
    SAI_CUDA_CHECK(cudaMemcpyAsync(d_ws + 2 * W, fl.data(), sizeof(int32_t) * 2 * W, cudaMemcpyHostToDevice, e->s_comp));
    SAI_CUDA_CHECK(cudaStreamSynchronize(e->s_comp));  // fl goes out of scope
  }
  uint32_t* d_mask_u = static_cast<uint32_t*>(e->mask.p);
  if (n_tiles > 0)
    if (int rc = sai_site_flags(&e->lay, e->packed.p, 0, n_tiles, n_tiles, jobs, n_jobs, d_mask_u,
                                d_mask_u + (size_t)n_jobs * n_tiles, static_cast<double*>(e->qval.p), stride, nullptr,
                                nullptr, 0, 0, e->s_comp))
      return rc;
  return run_windows(e, out);
}

}  // extern "C"

namespace sai {

// The group of blocks [b, b1) that starts at block b: at most slice_bytes of text together with the
// carried line and a newline (at least one block), so the ring slots are not reallocated slice after slice.
static int64_t vcf_group_end(const sai_engine* e, const int64_t* out_off, int64_t n_blocks, int64_t b) {
  const int64_t c = (int64_t)e->vcf.carry.size();
  int64_t b1 = b + 1;
  while (b1 < n_blocks && c + out_off[b1 + 1] - out_off[b] + 1 <= e->vcf.slice_bytes) ++b1;
  return b1;
}

// Group [b, b1) inflated by the staging threads straight into the slot behind the carried line; the
// incomplete last line is carried on.  `from`: text offset of the first record when it lies inside
// block b; `eof`: the group ends the file, so a last line without a newline is complete.
static int vcf_bgzf_group_host(sai_engine* e, const uint8_t* data, const int64_t* block_off, const int64_t* out_off,
                               int64_t b, int64_t b1, int64_t from, bool eof) {
  auto& V = e->vcf;
  const int64_t c = (int64_t)V.carry.size();
  const int64_t text = out_off[b1] - out_off[b];
  char* h = nullptr;
  if (int rc = vcf_acquire_slot(e, c + text + 1, &h)) return rc;
  if (c) memcpy(h, V.carry.data(), (size_t)c);
  const double t0 = now_s();
  constexpr int64_t kGroup = 16;  // blocks per task (~1 MB of text)
  std::atomic<int> bad_rc{SAI_OK};
  std::mutex msg_mu;
  std::string msg;
  const std::function<void(int64_t)> f = [&](int64_t i) {
    const int64_t g0 = b + i * kGroup, g1 = std::min(b1, g0 + kGroup);
    int64_t rel[kGroup + 1];
    for (int64_t k = g0; k <= g1; ++k) rel[k - g0] = out_off[k] - out_off[b] + c;
    const int rc = sai_bgzf_inflate(data, block_off + g0, rel, g1 - g0, reinterpret_cast<uint8_t*>(h), 1);
    if (rc != SAI_OK) {
      std::lock_guard<std::mutex> lk(msg_mu);
      if (bad_rc.load() == SAI_OK) msg = sai_last_error();
      bad_rc.store(rc);
    }
  };
  V.pool.run(stage_threads(e), (b1 - b + kGroup - 1) / kGroup, f);
  V.t_stage += now_s() - t0;
  if (bad_rc.load() != SAI_OK) {
    set_error("%s", msg.c_str());
    return bad_rc.load();
  }
  const int64_t lo = c == 0 && from > out_off[b] ? from - out_off[b] : 0;  // the header stays behind
  int64_t end = c + text;
  if (eof && end > lo && h[end - 1] != '\n') h[end++] = '\n';  // last line without a newline
  const void* nl = end > lo ? memrchr(h + lo, '\n', (size_t)(end - lo)) : nullptr;
  const int64_t cut = nl ? static_cast<const char*>(nl) - h + 1 : lo;
  std::vector<char> rest(h + cut, h + end);  // the incomplete last line, carried into the next slot
  if (cut > lo)
    if (int rc = vcf_launch_slot(e, lo, cut - lo)) return rc;
  V.carry.swap(rest);
  return SAI_OK;
}

// The compressed ring (pinned + device) with slots of at least `bytes`; grows after a drain.
static int vcf_comp_ring(sai_engine* e, size_t bytes) {
  auto& V = e->vcf;
  if (bytes <= V.comp_slot) return SAI_OK;  // comp_slot is 0 whenever the ring's depth changed
  SAI_CUDA_CHECK(cudaStreamSynchronize(e->s_copy));
  SAI_CUDA_CHECK(cudaStreamSynchronize(e->s_comp));
  const size_t slot = align256(std::max(bytes, std::max<size_t>(2 * V.comp_slot, 1u << 20)));
  if (V.h_comp) SAI_CUDA_CHECK(cudaFreeHost(V.h_comp));
  V.h_comp = nullptr;
  V.comp_slot = 0;
  SAI_CUDA_CHECK(cudaHostAlloc(reinterpret_cast<void**>(&V.h_comp), slot * V.ring, cudaHostAllocDefault));
  if (int rc = grow(e->vcomp, slot * V.ring)) return rc;
  V.comp_slot = slot;
  return SAI_OK;
}

// Group [b, b1) inflated on the device.  The host inflates only the boundary: the group's last block
// (and, when it holds no newline, the ones before it, up to kLookBack bytes of text) to find the last line
// end `cut`; the bytes behind it are the next group's carry.  The slot then holds [carry | text of the
// group's blocks] -- the carry travels as stored deflate pseudo-blocks in the same copy -- and [lo, cut)
// is parsed.  A group whose last kLookBack bytes hold no newline (a line of about that length or longer)
// is staged by vcf_bgzf_group_host.  The slot's text starts `pad` bytes in, so that the parsed range
// begins 16-byte aligned as the parse kernels read it.
static int vcf_bgzf_group_device(sai_engine* e, const uint8_t* data, const int64_t* block_off, const int64_t* out_off,
                                 int64_t b, int64_t b1, int64_t from, bool eof) {
  constexpr int64_t kLookBack = 1 << 20;
  auto& V = e->vcf;
  const int64_t c = (int64_t)V.carry.size();
  const int64_t text = out_off[b1] - out_off[b];
  const int64_t lo = c == 0 && from > out_off[b] ? from - out_off[b] : 0;
  const int64_t pad = (16 - (lo & 15)) & 15;
  const double t0 = now_s();
  std::vector<std::vector<char>> tail;  // text of blocks b1 - 1, b1 - 2, ..., k inflated by the host
  int64_t k = b1, cut = -1;
  bool newline = false;  // a '\n' pseudo-block completes the file's last line
  while (k > b && cut < 0 && out_off[b1] - out_off[k] < kLookBack) {
    --k;
    const int64_t isz = out_off[k + 1] - out_off[k];
    const int64_t at = c + out_off[k] - out_off[b];  // slot offset of block k
    tail.emplace_back((size_t)isz);
    std::vector<char>& blk = tail.back();
    if (isz > 0) {
      const int64_t rel[2] = {0, isz};
      if (sai_bgzf_inflate(data, block_off + k, rel, 1, reinterpret_cast<uint8_t*>(blk.data()), 1) != SAI_OK) {
        V.t_boundary += now_s() - t0;
        set_error("BGZF block %lld is corrupt", (long long)k);
        return SAI_E_CORRUPT;
      }
      if (eof) {  // the range ends at the end of the file: its last line is complete
        newline = blk.back() != '\n';
        cut = c + text + (newline ? 1 : 0);
      } else {
        const int64_t from_k = std::max<int64_t>(0, lo - at);
        const void* nl = from_k < isz ? memrchr(blk.data() + from_k, '\n', (size_t)(isz - from_k)) : nullptr;
        if (nl) cut = at + (static_cast<const char*>(nl) - blk.data()) + 1;
      }
    }
    if (at <= lo) break;  // nothing of the group's records lies before block k
  }
  if (cut < 0 && eof && c > lo && k == b) {  // only empty blocks behind the carried line: it is the file's last line
    cut = c + text + 1;
    newline = true;
  }
  V.t_boundary += now_s() - t0;
  if (eof && c + text <= lo) return SAI_OK;  // nothing behind the header
  if (cut <= lo) return vcf_bgzf_group_host(e, data, block_off, out_off, b, b1, from, eof);
  // descriptors, the group's members as they lie in the file, then the pseudo-blocks
  const int64_t n_real = b1 - b;
  const int64_t n_carry = (c + 65534) / 65535;
  const int64_t n_desc = n_real + n_carry + (newline ? 1 : 0);
  std::vector<sai_bgzf_block> desc((size_t)n_desc);
  const size_t desc_bytes = align256(sizeof(sai_bgzf_block) * (size_t)n_desc);
  if (int rc = sai_bgzf_descriptors(data, block_off + b, out_off + b, n_real, (int64_t)desc_bytes, pad + c, desc.data()))
    return rc;
  for (int64_t j = 0; j + 1 < n_real; ++j) {  // the members are copied as one span of the file
    const sai_bgzf_block& d = desc[(size_t)j];
    const int64_t member_end = d.comp_off + d.comp_bytes + 8 - (int64_t)desc_bytes;
    SAI_REQUIRE(block_off[b + j + 1] - block_off[b] == member_end, "sai_engine_vcf_feed_bgzf_device: blocks are not contiguous");
  }
  const int64_t span = desc[(size_t)n_real - 1].comp_off + desc[(size_t)n_real - 1].comp_bytes + 8 - (int64_t)desc_bytes;
  const int64_t pseudo = c + 5 * n_carry + (newline ? 6 : 0);
  const size_t bytes = desc_bytes + (size_t)span + (size_t)pseudo;
  char* h = nullptr;
  if (int rc = vcf_acquire_slot(e, pad + c + text + 1, &h)) return rc;
  if (int rc = vcf_comp_ring(e, align256(bytes) + sizeof(int32_t) * (size_t)n_desc)) return rc;
  uint8_t* hc = reinterpret_cast<uint8_t*>(V.h_comp) + (size_t)(V.n_slices % V.ring) * V.comp_slot;
  uint8_t* ps = hc + desc_bytes + span;
  int64_t ps_off = (int64_t)desc_bytes + span;
  auto stored = [&](int64_t idx, const char* src, int64_t len, int64_t text_off) {  // BFINAL, BTYPE 00, LEN, NLEN, bytes
    ps[0] = 1;
    ps[1] = (uint8_t)(len & 0xff), ps[2] = (uint8_t)(len >> 8);
    ps[3] = (uint8_t)(~len & 0xff), ps[4] = (uint8_t)((~len >> 8) & 0xff);
    memcpy(ps + 5, src, (size_t)len);
    sai_bgzf_block& d = desc[(size_t)idx];
    d.comp_off = ps_off;
    d.comp_bytes = (int32_t)(5 + len);
    d.text_off = text_off;
    d.isize = (int32_t)len;
    d.crc = sai_crc32(reinterpret_cast<const uint8_t*>(src), len, 0);
    ps += 5 + len;
    ps_off += 5 + len;
  };
  for (int64_t i = 0; i < n_carry; ++i) {
    const int64_t a = i * 65535, len = std::min<int64_t>(65535, c - a);
    stored(n_real + i, V.carry.data() + a, len, pad + a);
  }
  if (newline) stored(n_desc - 1, "\n", 1, pad + c + text);
  memcpy(hc, desc.data(), sizeof(sai_bgzf_block) * (size_t)n_desc);
  staged_copy(e, reinterpret_cast<char*>(hc + desc_bytes), reinterpret_cast<const char*>(data + block_off[b]), (size_t)span);
  const DevGroup g{bytes, n_desc, b};
  if (int rc = vcf_launch_slot(e, pad + lo, cut - lo, &g)) return rc;
  // the carry: slot bytes [cut, c + text) -- inside the blocks the host inflated (tail, last block first)
  std::vector<char> rest;
  if (!eof) {
    int64_t skip = cut - (c + out_off[k] - out_off[b]);
    rest.reserve((size_t)(c + text - cut));
    for (auto it = tail.rbegin(); it != tail.rend(); ++it) {
      const int64_t from_here = std::min<int64_t>(skip, (int64_t)it->size());
      rest.insert(rest.end(), it->begin() + from_here, it->end());
      skip -= from_here;
    }
  }
  V.carry.swap(rest);
  return SAI_OK;
}

}  // namespace sai

extern "C" {

static int vcf_feed_bgzf_impl(sai_engine* e, const uint8_t* data, const int64_t* block_off, const int64_t* out_off,
                              int64_t n_blocks, int64_t skip, int device, bool at_eof);
int sai_engine_vcf_feed_bgzf(sai_engine* e, const uint8_t* data, const int64_t* block_off, const int64_t* out_off,
                             int64_t n_blocks, int64_t skip) {
  const double t0 = now_s();
  const int rc = vcf_feed_bgzf_impl(e, data, block_off, out_off, n_blocks, skip, 0, true);
  if (e) e->vcf.t_feed += now_s() - t0;
  return rc;
}
int sai_engine_vcf_feed_bgzf_device(sai_engine* e, const uint8_t* data, const int64_t* block_off, const int64_t* out_off,
                                    int64_t n_blocks, int64_t skip, int32_t at_eof) {
  const double t0 = now_s();
  const int rc = vcf_feed_bgzf_impl(e, data, block_off, out_off, n_blocks, skip, 1, at_eof != 0);
  if (e) e->vcf.t_feed += now_s() - t0;
  return rc;
}
static int vcf_feed_bgzf_impl(sai_engine* e, const uint8_t* data, const int64_t* block_off, const int64_t* out_off,
                              int64_t n_blocks, int64_t skip, int device, bool at_eof) {
  SAI_REQUIRE(e && n_blocks >= 0 && skip >= 0 && (n_blocks == 0 || (data && block_off && out_off)),
              "sai_engine_vcf_feed_bgzf: bad argument");
  auto& V = e->vcf;
  SAI_REQUIRE(V.state == 1, "sai_engine_vcf_feed_bgzf: no ingest session (sai_engine_vcf_begin)");
  if (V.sticky_rc) return V.sticky_rc;
  if (n_blocks == 0) return SAI_OK;
  SAI_REQUIRE(out_off[0] == 0 && skip <= out_off[n_blocks], "sai_engine_vcf_feed_bgzf: bad text offsets");
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  // the block that holds text offset `skip`
  int64_t b = std::upper_bound(out_off, out_off + n_blocks + 1, skip) - out_off - 1;
  int64_t from = skip;  // first text offset of the records (inside block b)
  V.carry.clear();
  while (b < n_blocks) {
    const int64_t b1 = vcf_group_end(e, out_off, n_blocks, b);
    SAI_REQUIRE(out_off[b1] >= out_off[b], "sai_engine_vcf_feed_bgzf: text offsets are not monotonic");
    SAI_REQUIRE((int64_t)V.carry.size() + out_off[b1] - out_off[b] + 1 < (int64_t(1) << 31),
                "sai_engine_vcf_feed_bgzf: a line of more than 2 GB");
    const bool eof = at_eof && b1 == n_blocks;
    const int rc = device ? vcf_bgzf_group_device(e, data, block_off, out_off, b, b1, from, eof)
                          : vcf_bgzf_group_host(e, data, block_off, out_off, b, b1, from, eof);
    if (rc) {
      V.sticky_rc = rc;
      return rc;
    }
    b = b1;
    from = out_off[b];
  }
  return SAI_OK;
}

int sai_engine_vcf_stats(const sai_engine* e, double* out, int32_t n) {
  SAI_REQUIRE(e && out && n >= 0, "sai_engine_vcf_stats: bad argument");
  for (int i = 0; i < n && i < 14; ++i) out[i] = e->vcf.stats[i];
  return SAI_OK;
}

int sai_engine_set_vcf_slicing(sai_engine* e, int64_t slice_bytes, int32_t ring) {
  SAI_REQUIRE(e, "NULL engine");
  auto& V = e->vcf;
  SAI_REQUIRE(V.state != 1, "sai_engine_set_vcf_slicing: an ingest session is feeding");
  SAI_REQUIRE(slice_bytes <= 0 || (slice_bytes >= 64 && slice_bytes < (int64_t(1) << 30)), "slice size outside [64, 2^30)");
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  V.slice_bytes = slice_bytes > 0 ? slice_bytes : (32ll << 20);
  const int r = ring > 0 ? std::max(2, (int)ring) : 4;
  // new geometry: the slots are reallocated by the next slice
  SAI_CUDA_CHECK(cudaStreamSynchronize(e->s_copy));
  SAI_CUDA_CHECK(cudaStreamSynchronize(e->s_comp));
  if (V.h_ring) SAI_CUDA_CHECK(cudaFreeHost(V.h_ring));
  V.h_ring = nullptr;
  V.slot_bytes = 0;
  if (V.h_comp) SAI_CUDA_CHECK(cudaFreeHost(V.h_comp));  // the compressed ring has `ring` slots too
  V.h_comp = nullptr;
  V.comp_slot = 0;
  V.ring = r;
  return SAI_OK;
}

int64_t sai_engine_vcf_slices(const sai_engine* e) { return e ? e->vcf.n_slices : 0; }

int sai_engine_loaded_tiles(sai_engine* e, uint8_t* out, uint64_t cap) {
  SAI_REQUIRE(e && e->vcf.state == 2, "sai_engine_loaded_tiles: no finished ingest session");
  const uint64_t bytes = sai_packed_bytes(&e->lay, e->n_sites);
  SAI_REQUIRE(cap >= bytes && (bytes == 0 || out), "sai_engine_loaded_tiles: %llu bytes needed", (unsigned long long)bytes);
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  if (bytes) SAI_CUDA_CHECK(cudaMemcpy(out, e->packed.p, bytes, cudaMemcpyDeviceToHost));
  return SAI_OK;
}

int sai_engine_set_vcf_neg_table(sai_engine* e, int32_t on, int64_t min_entries) {
  SAI_REQUIRE(e, "NULL engine");
  SAI_REQUIRE(e->vcf.state != 1, "sai_engine_set_vcf_neg_table: an ingest session is feeding");
  SAI_REQUIRE(min_entries >= 0 && min_entries <= sai::kNegMaxEntries,
              "sai_engine_set_vcf_neg_table: min_entries %lld outside 0..2^31 - 1", (long long)min_entries);
  e->vcf.neg_on = on != 0;
  e->vcf.neg_min = min_entries;
  return SAI_OK;
}

int64_t sai_engine_loaded_neg_table(sai_engine* e, int64_t* neg_off, int32_t* site, int32_t* ind, int32_t* val,
                                    int64_t cap) {
  SAI_REQUIRE(e, "NULL engine");
  auto& V = e->vcf;
  SAI_REQUIRE(V.neg && V.neg_n >= 0, "sai_engine_loaded_neg_table: the last ingest session kept no negative-value table");
  if (V.state != 2) return V.neg_n;  // finished with SAI_E_CAPACITY: the count a repeat needs
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  if (neg_off) std::copy(V.neg_off.begin(), V.neg_off.end(), neg_off);
  const int64_t n = V.neg_n;
  if (cap >= n && n > 0 && site && ind && val) {
    const size_t part = align256(sizeof(int32_t) * (size_t)n);
    const char* t = static_cast<const char*>(e->vnegt.p);
    SAI_CUDA_CHECK(cudaMemcpy(site, t, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
    SAI_CUDA_CHECK(cudaMemcpy(ind, t + part, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
    SAI_CUDA_CHECK(cudaMemcpy(val, t + 2 * part, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
  }
  return n;
}

int sai_engine_dd_sums_loaded(sai_engine* e, int32_t ref_pop, int32_t tgt_pop, const int32_t* src_pops, int32_t n_src,
                              int64_t* ref_sum, int64_t* tgt_sum, int32_t m_max) {
  SAI_REQUIRE(e && e->vcf.state == 2 && e->n_jobs > 0, "sai_engine_dd_sums_loaded: no scored ingest session");
  SAI_REQUIRE(ref_sum && tgt_sum && src_pops, "NULL argument");
  auto& V = e->vcf;
  SAI_REQUIRE(V.neg, "sai_engine_dd_sums_loaded: the ingest session kept no negative-value table");
  SAI_REQUIRE(!e->pieces.empty() || !V.genome || V.gq.n_chrom == 1,
              "sai_engine_dd_sums_loaded: a genome session is scored in pieces");
  // each piece's row of the table: a genome session's piece is the chromosome whose sites it covers
  // (the table's sites are chromosome-local); one chunk is the only row
  std::vector<std::array<int64_t, 5>> P;
  for (const auto& q : scored_pieces(e)) {
    int64_t c = e->pieces.empty() ? 0 : -1;
    for (size_t k = 0; k < V.chrom_sites.size() && c < 0; ++k)
      if (V.chrom_sites[k][0] == q[2] && V.chrom_sites[k][1] == q[3]) c = (int64_t)k;
    SAI_REQUIRE(c >= 0 || q[3] == 0, "sai_engine_dd_sums_loaded: piece at site %lld (%lld sites) is not a chromosome",
                (long long)q[2], (long long)q[3]);
    P.push_back({q[0], q[1], q[2], q[3], c});
  }
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  const size_t part = align256(sizeof(int32_t) * (size_t)std::max<int64_t>(V.neg_n, 1));
  const char* t = static_cast<const char*>(e->vnegt.p);
  return dd_sums_impl(e, &e->lay, ref_pop, tgt_pop, src_pops, n_src, m_max, reinterpret_cast<const int32_t*>(t),
                      reinterpret_cast<const int32_t*>(t + part), reinterpret_cast<const int32_t*>(t + 2 * part),
                      V.neg_off.data(), P, ref_sum, tgt_sum);
}

}  // extern "C"

int sai_engine_format_scores(sai_engine* e, const sai_format_input* in, int64_t* sizes) {
  SAI_REQUIRE(e, "NULL engine");
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  return sai::format_scores(e->fmt, in, e->s_comp, sizes);
}

int sai_engine_format_text(sai_engine* e, int32_t which, char* out, int64_t cap) {
  SAI_REQUIRE(e, "NULL engine");
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  return sai::format_text(e->fmt, which, out, cap, e->s_comp);
}

int sai_engine_format_stats(const sai_engine* e, double* out, int32_t n) {
  SAI_REQUIRE(e, "NULL engine");
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  return sai::format_stats(const_cast<sai_engine*>(e)->fmt, out, n);
}

int sai_engine_format_doubles(sai_engine* e, const double* x, int64_t n, char* out) {
  SAI_REQUIRE(e, "NULL engine");
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  return sai::format_doubles_device(x, n, out, e->s_comp);
}

int sai_engine_table_load(sai_engine* e, const char* text, int64_t n_bytes, int32_t n_cols, int64_t chunk_rows,
                          int64_t* info) {
  SAI_REQUIRE(e, "NULL engine");
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  return sai::table_load(e->tab, text, n_bytes, n_cols, chunk_rows, info, e->s_comp);
}

int sai_engine_table_classes(sai_engine* e, uint32_t* out, int64_t cap) {
  SAI_REQUIRE(e, "NULL engine");
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  return sai::table_classes(e->tab, out, cap, e->s_comp);
}

int sai_engine_table_parse(sai_engine* e, const int32_t* kinds, int32_t first_metric, int32_t chrom, int32_t start,
                           int32_t end, double* d_vals, double* first_val, int64_t* n_runs) {
  SAI_REQUIRE(e, "NULL engine");
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  return sai::table_parse(e->tab, kinds, first_metric, chrom, start, end, d_vals, first_val, n_runs, e->s_comp);
}

int sai_engine_table_runs(sai_engine* e, int64_t* off, int64_t* len, int64_t cap) {
  SAI_REQUIRE(e, "NULL engine");
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  return sai::table_runs(e->tab, off, len, cap, e->s_comp);
}

int sai_engine_table_order(sai_engine* e, const int32_t* run_rank, int64_t n_runs) {
  SAI_REQUIRE(e, "NULL engine");
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  return sai::table_order(e->tab, run_rank, n_runs, e->s_comp);
}

int sai_engine_table_build(sai_engine* e, const double* thr, const int32_t* strict, int64_t* offsets) {
  SAI_REQUIRE(e, "NULL engine");
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  return sai::table_build(e->tab, thr, strict, offsets, e->s_comp);
}

int sai_engine_table_text(sai_engine* e, char* out, int64_t cap) {
  SAI_REQUIRE(e, "NULL engine");
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  return sai::table_text(e->tab, out, cap, e->s_comp);
}

int sai_engine_table_stats(const sai_engine* e, double* out, int32_t n) {
  SAI_REQUIRE(e, "NULL engine");
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  return sai::table_stats(const_cast<sai_engine*>(e)->tab, out, n);
}

int sai_engine_parse_doubles(sai_engine* e, const char* text, const int64_t* offs, int64_t n, double* out, uint8_t* ok) {
  SAI_REQUIRE(e, "NULL engine");
  SAI_CUDA_CHECK(cudaSetDevice(e->device));
  return sai::parse_doubles_device(text, offs, n, out, ok, e->s_comp);
}
