// Sanitizer fuzz of the BGZF block decoders -- the host one (sai_b200/csrc/inflate_fast.cpp) and the
// host build of the device one (sai_b200/csrc/inflate_device.cuh, one lane): valid streams of every
// zlib level / strategy must decode exactly (and the device decoder's CRC-32 must equal zlib's, also
// when split over 32 lanes or a random lane count and combined);
// bit-flipped, truncated and randomised streams must be refused or decoded WITHOUT touching memory
// outside the exact-size heap buffers.
//   g++ -O1 -g -fsanitize=address,undefined -std=c++17 tools/inflate_fuzz.cpp sai_b200/csrc/inflate_fast.cpp -lz -o tools/bin/inflate_fuzz && tools/bin/inflate_fuzz
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include <zlib.h>
#include "../sai_b200/csrc/inflate_fast.h"
#include "../sai_b200/csrc/inflate_device.cuh"
static uint32_t crc_tab[256];
static sai::infl::Tables tabs;
static int device_decoder(const uint8_t* in, size_t n, uint8_t* out, size_t on, uint32_t* crc) {
  const sai::infl::Team t{0, 1};
  const int st = sai::infl::inflate_block(in, (uint32_t)n, out, (uint32_t)on, tabs, t);
  *crc = sai::infl::crc_finish(sai::infl::crc_share(out, (uint32_t)on, crc_tab, t), (uint32_t)on);
  return st;
}
// The CRC of a team of `width` lanes: every lane's share of [p, p + n), combined in GF(2).
static uint32_t team_crc(const uint8_t* p, size_t n, int width) {
  uint32_t shares = 0;
  for (int lane = 0; lane < width; ++lane) shares ^= sai::infl::crc_share(p, (uint32_t)n, crc_tab, {lane, width});
  return sai::infl::crc_finish(shares, (uint32_t)n);
}
int main() {
  for (uint32_t i = 0; i < 256; ++i) crc_tab[i] = sai::infl::crc_table_entry(i);
  long dev_refused = 0, dev_accepted = 0;
  srand(7);
  long refused = 0, accepted = 0, same = 0;
  for (int round = 0; round < 400; ++round) {
    // build a source buffer: mix of text-like runs and noise
    size_t n = 1 + rand() % 70000;
    std::vector<uint8_t> src(n);
    int mode = rand() % 4;
    for (size_t i = 0; i < n; ++i) src[i] = mode == 0 ? (uint8_t)rand() : mode == 1 ? (uint8_t)("0|0\t"[i & 3]) ^ ((rand() % 50 == 0) ? 1 : 0) : mode == 2 ? (uint8_t)(rand() % 3 + 'a') : (uint8_t)((i / 97) & 0xff);
    std::vector<uint8_t> comp(compressBound(n) + 64);
    z_stream zs; memset(&zs, 0, sizeof zs);
    int level = rand() % 10, strat = (rand() % 5 == 0) ? Z_FIXED : (rand() % 7 == 0 ? Z_HUFFMAN_ONLY : rand() % 6 == 0 ? Z_RLE : rand() % 5 == 0 ? Z_FILTERED : Z_DEFAULT_STRATEGY);
    deflateInit2(&zs, level, Z_DEFLATED, -15, 9, strat);
    zs.next_in = src.data(); zs.avail_in = n; zs.next_out = comp.data(); zs.avail_out = comp.size();
    deflate(&zs, Z_FINISH); size_t cn = zs.total_out; deflateEnd(&zs);
    // exact-size heap buffers so that ASAN sees any out-of-range access
    {
      uint8_t* in = (uint8_t*)malloc(cn); memcpy(in, comp.data(), cn);
      uint8_t* out = (uint8_t*)malloc(n);
      if (!sai::inflate_raw(in, cn, out, n) || memcmp(out, src.data(), n)) { printf("MISMATCH on valid stream n=%zu level=%d strat=%d\n", n, level, strat); return 1; }
      if (n <= 65536) {  // a BGZF block's text: what the device decoder takes
        memset(out, 0, n);
        uint32_t crc = 0;
        if (device_decoder(in, cn, out, n, &crc) != 0 || memcmp(out, src.data(), n) || crc != crc32(0, src.data(), n)) {
          printf("DEVICE DECODER MISMATCH on valid stream n=%zu level=%d strat=%d\n", n, level, strat); return 1;
        }
        if (team_crc(out, n, 32) != crc || team_crc(out, n, 1 + rand() % 31) != crc) {
          printf("TEAM CRC MISMATCH n=%zu\n", n); return 1;
        }
      }
      ++same; free(in); free(out);
    }
    for (int k = 0; k < 60; ++k) {
      size_t m = cn; int kind = rand() % 3;
      if (kind == 1) m = rand() % (cn + 1);
      uint8_t* in = (uint8_t*)malloc(m ? m : 1); memcpy(in, comp.data(), m);
      if (kind == 0 && m) for (int f = 0; f < 1 + rand() % 3; ++f) in[rand() % m] ^= 1 << (rand() % 8);
      if (kind == 2 && m) { size_t at = rand() % m; for (size_t i = at; i < m; ++i) in[i] = (uint8_t)rand(); }
      size_t on = (rand() % 4 == 0) ? (size_t)(rand() % 70000) : n;
      uint8_t* out = (uint8_t*)malloc(on ? on : 1);
      if (sai::inflate_raw(in, m, out, on)) ++accepted; else ++refused;
      uint32_t crc = 0;
      if (on <= 65536) { if (device_decoder(in, m, out, on, &crc) == 0) ++dev_accepted; else ++dev_refused; }
      free(in); free(out);
    }
  }
  printf("valid %ld, corrupted: refused %ld accepted %ld; device decoder: refused %ld accepted %ld\n", same, refused,
         accepted, dev_refused, dev_accepted);
  return 0;
}
