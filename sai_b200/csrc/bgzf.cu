// Host-side BGZF (bgzip) reader for the VCF ingest (N2).  No device code in this file.
//
// The reference reads `.vcf.gz` through scikit-allel / pysam (htslib).  A bgzip file is a
// sequence of independent gzip members of at most 64 KB ("blocks", SAM spec section 4.1): a
// gzip header whose extra field carries the subfield 'B','C' = total block size - 1, raw
// deflate data, CRC32 and ISIZE.  Independent blocks inflate in parallel, which turns the
// single-threaded decompression (the slowest stage of ingest once the parser runs at GB/s)
// into a multi-threaded one.
#include <string.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <new>
#include <thread>
#include <vector>

#include "common.cuh"
#include "inflate_fast.h"
#include "vcf_parse.h"

namespace sai {

static inline uint32_t le16(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }
static inline uint32_t le32(const uint8_t* p) { return le16(p) | (le16(p + 2) << 16); }

// total size of the block at p (0: not a complete / valid BGZF block within `avail` bytes);
// *payload_off = where its raw deflate data starts (behind the whole FEXTRA field); the one walk of the
// gzip header, also behind the device inflater's descriptors (sai_bgzf_descriptors)
static int64_t bgzf_block_size(const uint8_t* p, int64_t avail, int64_t* payload_off) {
  if (avail < 18) return 0;
  if (p[0] != 31 || p[1] != 139 || p[2] != 8 || !(p[3] & 4)) return -1;
  const int64_t xlen = le16(p + 10);
  if (avail < 12 + xlen) return 0;
  const uint8_t* x = p + 12;
  const uint8_t* xe = x + xlen;
  int64_t bsize = -1;
  while (x + 4 <= xe) {
    const int64_t slen = le16(x + 2);
    if (x[0] == 'B' && x[1] == 'C' && slen == 2 && x + 6 <= xe) bsize = (int64_t)le16(x + 4) + 1;
    x += 4 + slen;
  }
  if (bsize < 0) return -1;
  if (bsize < 12 + xlen + 8) return -1;
  if (avail < bsize) return 0;
  *payload_off = 12 + xlen;
  return bsize;
}

// Inflates the (scan-validated) block at p into exactly `want` bytes: the in-house decoder first
// (inflate_fast.cpp: ~3x zlib on VCF text); whatever it does not accept, or whose CRC-32 does not
// match, is decoded again by zlib (`zs`: an inflateInit2(-15) stream of the calling thread) before
// the block is called corrupt.
static bool inflate_one(const uint8_t* p, uint8_t* out, int64_t want, z_stream* zs) {
  int64_t payload = 0;
  const int64_t bs = bgzf_block_size(p, (int64_t)1 << 20, &payload);
  if (bs <= 0) return false;
  if (want == 0) return true;  // empty block (the EOF marker)
  const uint32_t want_crc = le32(p + bs - 8);
  if (inflate_raw(p + payload, (size_t)(bs - payload - 8), out, (size_t)want) && crc32_fast(out, (size_t)want, 0) == want_crc)
    return true;
  inflateReset(zs);
  zs->next_in = const_cast<Bytef*>(p + payload);
  zs->avail_in = (uInt)(bs - payload - 8);
  zs->next_out = out;
  zs->avail_out = (uInt)want;
  return inflate(zs, Z_FINISH) == Z_STREAM_END && (int64_t)zs->total_out == want &&
         crc32(crc32(0L, Z_NULL, 0), out, (uInt)want) == want_crc;
}

}  // namespace sai

using namespace sai;

extern "C" {

int32_t sai_is_bgzf(const uint8_t* data, int64_t len) {
  int64_t off = 0;
  return data && bgzf_block_size(data, len, &off) > 0 ? 1 : 0;
}

int64_t sai_bgzf_scan(const uint8_t* data, int64_t len, int64_t max_blocks, int64_t max_out_bytes,
                      int64_t* block_off, int64_t* out_off, int64_t* consumed) {
  if (!data || len < 0 || max_blocks < 0 || !block_off || !out_off || !consumed) {
    set_error("sai_bgzf_scan: bad argument");
    return SAI_E_ARG;
  }
  int64_t at = 0, n = 0, out = 0;
  out_off[0] = 0;
  while (n < max_blocks && at < len) {
    int64_t payload = 0;
    const int64_t bs = bgzf_block_size(data + at, len - at, &payload);
    if (bs < 0) {
      set_error("not a BGZF block at offset %lld", (long long)at);
      return SAI_E_ARG;
    }
    if (bs == 0) break;  // incomplete block: the caller supplies more bytes
    const int64_t isize = le32(data + at + bs - 4);
    if (isize > (1 << 16)) {  // SAM spec 4.1: at most 64 KB of text per block
      set_error("BGZF block at offset %lld claims %lld bytes of text", (long long)at, (long long)isize);
      return SAI_E_ARG;
    }
    if (n > 0 && out + isize > max_out_bytes) break;
    block_off[n] = at;
    out += isize;
    out_off[++n] = out;
    at += bs;
  }
  *consumed = at;
  return n;
}

int sai_bgzf_descriptors(const uint8_t* data, const int64_t* block_off, const int64_t* out_off, int64_t n_blocks,
                         int64_t comp_base, int64_t text_base, sai_bgzf_block* out) {
  if (!data || n_blocks < 0 || (n_blocks > 0 && (!block_off || !out_off || !out))) {
    set_error("sai_bgzf_descriptors: bad argument");
    return SAI_E_ARG;
  }
  for (int64_t j = 0; j < n_blocks; ++j) {
    int64_t payload = 0;
    const int64_t bs = bgzf_block_size(data + block_off[j], (int64_t)1 << 20, &payload);
    const int64_t isize = out_off[j + 1] - out_off[j];
    if (bs <= 0 || isize < 0 || isize > (1 << 16)) {
      set_error("sai_bgzf_descriptors: no BGZF block of <= 64 KB of text at offset %lld", (long long)block_off[j]);
      return SAI_E_ARG;
    }
    sai_bgzf_block& d = out[j];
    d.comp_off = comp_base + (block_off[j] - block_off[0]) + payload;
    d.text_off = text_base + out_off[j] - out_off[0];
    d.comp_bytes = (int32_t)(bs - payload - 8);
    d.isize = (int32_t)isize;
    d.crc = le32(data + block_off[j] + bs - 8);
    d.pad_ = 0;
  }
  return SAI_OK;
}

int sai_bgzf_inflate(const uint8_t* data, const int64_t* block_off, const int64_t* out_off, int64_t n_blocks,
                     uint8_t* out, int32_t n_threads) {
  if (!data || !block_off || !out_off || n_blocks < 0 || (n_blocks > 0 && !out)) {
    set_error("sai_bgzf_inflate: bad argument");
    return SAI_E_ARG;
  }
  if (n_threads <= 0) n_threads = (int)std::max(1u, std::thread::hardware_concurrency());
  n_threads = (int)std::min<int64_t>(n_threads, std::max<int64_t>(1, n_blocks / 4));
  std::atomic<int64_t> next{0};
  std::atomic<int64_t> bad{-1};
  auto work = [&]() {
    z_stream zs;
    memset(&zs, 0, sizeof(zs));
    if (inflateInit2(&zs, -15) != Z_OK) {
      bad.store(0);
      return;
    }
    for (;;) {
      const int64_t b0 = next.fetch_add(16);
      if (b0 >= n_blocks || bad.load(std::memory_order_relaxed) >= 0) break;
      const int64_t b1 = std::min(n_blocks, b0 + 16);
      for (int64_t b = b0; b < b1; ++b) {
        const int64_t want = out_off[b + 1] - out_off[b];
        const bool ok = inflate_one(data + block_off[b], out + out_off[b], want, &zs);
        if (!ok) {
          bad.store(b);
          break;
        }
      }
    }
    inflateEnd(&zs);
  };
  if (n_threads <= 1) {
    work();
  } else {
    std::vector<std::thread> th;
    for (int i = 0; i < n_threads; ++i) th.emplace_back(work);
    for (auto& t : th) t.join();
  }
  if (bad.load() >= 0) {
    set_error("BGZF block %lld is corrupt", (long long)bad.load());
    return SAI_E_ARG;
  }
  return SAI_OK;
}

// Fused bgzip read (see include/sai_b200.h).  Blocks are taken in groups of `group_blocks`; a
// thread inflates a group into its own buffer -- plus as many following blocks as it takes to
// complete the line that crosses the group's end -- and parses, right away and out of its cache,
// every line that STARTS inside the group (after the group's first byte, up to and including its
// end: a line starting exactly at the end belongs to this group, so the next group begins after
// its first newline).  The text never exists as a whole; rows are gathered in group order.
int64_t sai_bgzf_parse_gt(const uint8_t* data, const int64_t* block_off, const int64_t* out_off, int64_t n_blocks,
                          int64_t skip, const char* chrom, int64_t start, int64_t end, const int32_t* sample_column,
                          const int32_t* sample_ploidy, int32_t n_out, const int32_t* anc_pos, const char* anc_allele,
                          int64_t n_anc, int32_t* out_pos, int8_t* out_gt, int64_t row_stride, int64_t rows_cap,
                          int32_t group_blocks, int32_t n_threads) {
  if (!data || !block_off || !out_off || n_blocks < 0 || skip < 0 || !chrom || !sample_column || !sample_ploidy || n_out < 1 ||
      !out_pos || !out_gt || row_stride < n_out || rows_cap < 0 || (n_anc > 0 && (!anc_pos || !anc_allele))) {
    set_error("sai_bgzf_parse_gt: bad argument");
    return SAI_E_ARG;
  }
  GtParser P;
  if (!P.init(chrom, start, end, sample_column, sample_ploidy, n_out, anc_pos, anc_allele, n_anc)) {
    set_error("sai_bgzf_parse_gt: bad sample column / ploidy");
    return SAI_E_ARG;
  }
  if (n_blocks == 0) return 0;
  for (int64_t b = 0; b < n_blocks; ++b)  // SAM spec 4.1: a block holds at most 64 KB of text
    if (out_off[b + 1] < out_off[b] || out_off[b + 1] - out_off[b] > (1 << 16)) {
      set_error("BGZF block %lld claims %lld bytes of text", (long long)b, (long long)(out_off[b + 1] - out_off[b]));
      return SAI_E_ARG;
    }
  const int64_t G = group_blocks > 0 ? group_blocks : 16;  // ~1 MB of text: stays in the core's L2
  const int64_t n_groups = (n_blocks + G - 1) / G;
  if (n_threads <= 0) n_threads = (int)std::max(1u, std::thread::hardware_concurrency());
  n_threads = (int)std::min<int64_t>(n_threads, n_groups);
  std::vector<GtParser::SegOut> seg_out(n_groups);
  std::atomic<int64_t> next{0};
  std::atomic<int64_t> bad{-1};
  std::atomic<int> oom{0};
  auto work = [&]() {
    z_stream zs;
    memset(&zs, 0, sizeof(zs));
    if (inflateInit2(&zs, -15) != Z_OK) {
      bad.store(0);
      return;
    }
    GtParser::Scratch sc;
    std::vector<uint8_t> text;
    try {
    for (;;) {
      const int64_t g = next.fetch_add(1);
      if (g >= n_groups || bad.load(std::memory_order_relaxed) >= 0) break;
      const int64_t b0 = g * G, b1 = std::min(n_blocks, b0 + G);
      const int64_t own = out_off[b1] - out_off[b0];  // text bytes of the group's own blocks
      if (text.size() < (size_t)own + 2) text.resize((size_t)own + (1 << 17));
      bool ok = true;
      for (int64_t b = b0; b < b1 && ok; ++b) {
        ok = inflate_one(data + block_off[b], text.data() + (out_off[b] - out_off[b0]), out_off[b + 1] - out_off[b], &zs);
        if (!ok) bad.store(b);
      }
      if (!ok) break;
      // Where this group's lines begin.  Line starts are `skip` (the first record, absolute text
      // offset) and every position behind a newline after it; a group takes the starts s with
      // group_begin < s <= group_end (group 0 also s == 0).
      const int64_t rel_skip = skip - (out_off[b0] - out_off[0]);
      if (rel_skip > own) continue;  // still inside the header
      int64_t first;
      if (g == 0 || rel_skip > 0) {
        first = std::max<int64_t>(rel_skip, 0);  // the first record starts in this group
      } else {
        const void* nl = own > 0 ? memchr(text.data(), '\n', (size_t)own) : nullptr;
        if (!nl) continue;  // no line starts inside this group
        first = static_cast<const uint8_t*>(nl) - text.data() + 1;
      }
      // the end of the last line that starts at or before `own`: the first newline at index >= own,
      // which may need further blocks
      int64_t have = own, e = b1;
      int64_t limit = -1;
      for (;;) {
        const void* nl = have > own ? memchr(text.data() + own, '\n', (size_t)(have - own)) : nullptr;
        if (nl) {
          limit = static_cast<const uint8_t*>(nl) - text.data() + 1;
          break;
        }
        if (e >= n_blocks) break;
        const int64_t add = out_off[e + 1] - out_off[e];
        if (text.size() < (size_t)(have + add) + 2) text.resize((size_t)(have + add) + (1 << 17));
        if (!inflate_one(data + block_off[e], text.data() + have, add, &zs)) {
          bad.store(e);
          ok = false;
          break;
        }
        have += add;
        ++e;
      }
      if (!ok) break;
      if (limit < 0) {  // the file ends inside the last line: it is complete by definition
        if (have > 0 && text[have - 1] != '\n') text[have++] = '\n';
        limit = have;
      }
      if (first >= limit) continue;
      P.scan(reinterpret_cast<const char*>(text.data()) + first, reinterpret_cast<const char*>(text.data()) + limit, seg_out[g], sc);
      // the records point into `text`, which the next group overwrites: only pos and the rows survive
      for (auto& k : seg_out[g].kept) k.samples = k.line = nullptr;
    }
    } catch (const std::bad_alloc&) {
      oom.store(1);
      bad.store(0);  // stops the other threads
    }
    inflateEnd(&zs);
  };
  if (n_threads <= 1) {
    work();
  } else {
    std::vector<std::thread> th;
    for (int i = 0; i < n_threads; ++i) th.emplace_back(work);
    for (auto& t : th) t.join();
  }
  if (oom.load()) {
    set_error("sai_bgzf_parse_gt: out of host memory");
    return SAI_E_NOMEM;
  }
  if (bad.load() >= 0) {
    set_error("BGZF block %lld is corrupt", (long long)bad.load());
    return SAI_E_ARG;
  }
  const KeptLine* dropped = nullptr;
  const int64_t n_rows = P.gather(seg_out, out_pos, out_gt, row_stride, rows_cap, n_threads, &dropped);
  if (dropped) {
    set_error("sai_bgzf_parse_gt: more than %lld records", (long long)rows_cap);
    return SAI_E_CAPACITY;
  }
  return n_rows;
}

// A plain (single-member) gzip file in one go: RFC 1952 header, raw deflate stream, CRC-32 + ISIZE.
int64_t sai_gzip_inflate(const uint8_t* data, int64_t len, uint8_t* out, int64_t out_cap) {
  if (!data || len < 18 || out_cap < 0 || (out_cap > 0 && !out)) {
    set_error("sai_gzip_inflate: bad argument");
    return SAI_E_ARG;
  }
  if (data[0] != 31 || data[1] != 139 || data[2] != 8 || (data[3] & 0xe0)) {
    set_error("not a gzip file");
    return SAI_E_ARG;
  }
  const int flg = data[3];
  int64_t at = 10;
  if (flg & 4) {  // FEXTRA
    if (at + 2 > len) return SAI_E_ARG;
    at += 2 + (int64_t)le16(data + at);
  }
  for (int bit : {8, 16})  // FNAME, FCOMMENT: zero-terminated
    if (flg & bit) {
      const void* z = at < len ? memchr(data + at, 0, (size_t)(len - at)) : nullptr;
      if (!z) return SAI_E_ARG;
      at = static_cast<const uint8_t*>(z) - data + 1;
    }
  if (flg & 2) at += 2;  // FHCRC
  if (at + 8 > len) {
    set_error("truncated gzip file");
    return SAI_E_ARG;
  }
  const int64_t isize = le32(data + len - 4);  // of a single-member file below 4 GB of text
  if (isize > out_cap) {
    set_error("gzip file holds %lld bytes, buffer has %lld", (long long)isize, (long long)out_cap);
    return SAI_E_CAPACITY;
  }
  size_t used = 0;
  if (!inflate_raw(data + at, (size_t)(len - at - 8), out, (size_t)isize, &used) || (int64_t)used != len - at - 8 ||
      crc32_fast(out, (size_t)isize, 0) != le32(data + len - 8)) {
    set_error("not a single-member gzip file the fast decoder handles (several members, > 4 GB, or corrupt)");
    return SAI_E_DOMAIN;
  }
  return isize;
}

int32_t sai_inflate_raw(const uint8_t* in, int64_t in_len, uint8_t* out, int64_t out_len) {
  if (!in || in_len < 0 || out_len < 0 || (out_len > 0 && !out)) return 0;
  return inflate_raw(in, (size_t)in_len, out, (size_t)out_len) ? 1 : 0;
}

uint32_t sai_crc32(const uint8_t* data, int64_t len, int32_t isa) {
  return data && len > 0 ? crc32_fast(data, (size_t)len, isa) : 0u;
}

}  // extern "C"
