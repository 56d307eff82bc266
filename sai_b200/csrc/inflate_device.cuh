// Per-block raw-deflate decoder (RFC 1951) and CRC-32 of the device inflater (inflate_device.cu).
//
// The same code runs as one warp per BGZF block on the GPU and as plain C++ on the host, where
// tools/inflate_fuzz.cpp drives it under AddressSanitizer / UBSan.  A `Team` is the warp (32
// lanes) on the device and a single lane on the host: the bit reader, the symbol decode and every
// decision are lane-uniform (all lanes read the same bits and take the same branches); lane 0
// writes the literals and the tables' serial parts, and the whole team expands stored runs, match
// copies, the fast-table fill and the CRC.  A lane's share of a team loop is `for (k = lane; k < n;
// k += width)`: the same indices as the one-lane loop the fuzz runs, split between the lanes.  Reads stay inside [in, in + in_len), writes inside
// [out, out + out_len): a stream that wants more output, ends early or holds an invalid code is
// refused, never followed.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define SAI_HD __host__ __device__ __forceinline__
#else
#define SAI_HD inline
#endif

namespace sai {
namespace infl {

enum { kOk = 0, kBadStream = 1, kBadSize = 2, kBadCrc = 3 };

constexpr int kFastBits = 9;  // codes up to 9 bits decode with one table look-up

struct Huff {
  uint16_t count[16];                // codes of each length
  uint16_t offs[16];                 // index of the first symbol of each length in `symbol`
  uint16_t symbol[288];              // symbols ordered by (length, value)
  uint16_t fast[1 << kFastBits];     // (symbol << 4) | length of the code in the low bits, 0: longer
  uint16_t at[16];                   // build scratch: next free index of each length in `symbol`
};

struct Tables {
  Huff lit, dist;
  uint8_t lens[320];                 // code lengths of a dynamic block (286 + 30, 19 for the code-length code)
};

struct Team {
  int lane, width;
  SAI_HD void sync() const {
#ifdef __CUDA_ARCH__
    __syncwarp();
#endif
  }
  SAI_HD int bcast(int v) const {
#ifdef __CUDA_ARCH__
    return __shfl_sync(0xffffffffu, v, 0);
#else
    return v;
#endif
  }
};

struct BitReader {
  const uint8_t* in;
  uint32_t n, pos;
  uint64_t buf;
  int cnt;
  SAI_HD void refill() {
    while (cnt <= 56 && pos < n) {
      buf |= (uint64_t)in[pos++] << cnt;
      cnt += 8;
    }
  }
  SAI_HD bool need(int k) {
    if (cnt < k) refill();
    return cnt >= k;
  }
  SAI_HD uint32_t take(int k) {  // k <= 32, need(k) held
    const uint32_t v = (uint32_t)(buf & ((1ull << k) - 1));
    buf >>= k;
    cnt -= k;
    return v;
  }
};

// Canonical Huffman code of `n` symbols with code lengths len[0, n) (shared by the team) into h.
// Over-subscribed lengths are refused; an incomplete code is kept (its unused codes fail to decode).
SAI_HD bool build(Huff& h, const uint8_t* len, int n, const Team& t) {
  int ok = 1;
  if (t.lane == 0) {
    for (int l = 0; l < 16; ++l) h.count[l] = 0;
    for (int s = 0; s < n; ++s) h.count[len[s]]++;
    h.count[0] = 0;
    int left = 1;
    for (int l = 1; l < 16 && ok; ++l) {
      left = (left << 1) - h.count[l];
      if (left < 0) ok = 0;
    }
    h.offs[1] = 0;
    for (int l = 1; l < 15; ++l) h.offs[l + 1] = h.offs[l] + h.count[l];
    for (int l = 0; l < 16; ++l) h.at[l] = h.offs[l];
    for (int s = 0; s < n; ++s)
      if (len[s]) h.symbol[h.at[len[s]]++] = (uint16_t)s;
  }
  for (int i = t.lane; i < (1 << kFastBits); i += t.width) h.fast[i] = 0;
  t.sync();
  ok = t.bcast(ok);
  if (!ok) return false;
  // fast table: symbol i of the ordered list has the canonical code first[l] + (i - offs[l])
  int n_coded = 0;
  for (int l = 1; l <= kFastBits; ++l) n_coded += h.count[l];
  for (int i = t.lane; i < n_coded; i += t.width) {
    int l = 1;
    while (i >= h.offs[l] + h.count[l]) ++l;
    uint32_t code = 0;
    for (int k = 1; k <= l; ++k) code = (code + (k > 1 ? h.count[k - 1] : 0)) << 1;
    code += (uint32_t)(i - h.offs[l]);  // first[l] + rank
    uint32_t rev = 0;
    for (int k = 0; k < l; ++k) rev |= ((code >> k) & 1u) << (l - 1 - k);
    const uint16_t e = (uint16_t)((h.symbol[i] << 4) | l);
    for (uint32_t j = rev; j < (1u << kFastBits); j += 1u << l) h.fast[j] = e;
  }
  t.sync();
  return true;
}

// Next symbol of code h, or -1 (invalid code or not enough input).
SAI_HD int decode(const Huff& h, BitReader& br) {
  br.refill();
  const uint32_t peek = (uint32_t)br.buf;
  const uint16_t e = h.fast[peek & ((1u << kFastBits) - 1)];
  if (e) {
    const int l = e & 15;
    if (l > br.cnt) return -1;
    br.take(l);
    return e >> 4;
  }
  int code = 0, first = 0, index = 0;
  for (int l = 1; l < 16; ++l) {
    code |= (peek >> (l - 1)) & 1;
    const int count = h.count[l];
    if (code - first < count) {
      if (l > br.cnt) return -1;
      br.take(l);
      return h.symbol[index + code - first];
    }
    index += count;
    first = (first + count) << 1;
    code <<= 1;
  }
  return -1;
}

// literal/length and distance symbols of one compressed block until end-of-block
SAI_HD int codes(Tables& T, BitReader& br, uint8_t* out, uint32_t out_len, uint32_t& op, const Team& t) {
  for (;;) {
    int sym = decode(T.lit, br);
    if (sym < 0) return kBadStream;
    if (sym < 256) {
      if (op >= out_len) return kBadSize;
      if (t.lane == 0) out[op] = (uint8_t)sym;
      ++op;
      continue;
    }
    if (sym == 256) return kOk;
    sym -= 257;
    if (sym >= 29) return kBadStream;
    // RFC 1951 3.2.5: lengths 3..258 and distances 1..32768 from a base and extra bits
    int extra = sym < 8 || sym == 28 ? 0 : (sym >> 2) - 1;
    const uint32_t base = sym < 8 ? 3 + sym : sym == 28 ? 258 : ((4u + (sym & 3)) << extra) + 3;
    if (!br.need(extra)) return kBadStream;
    const uint32_t len = base + br.take(extra);
    const int ds = decode(T.dist, br);
    if (ds < 0 || ds >= 30) return kBadStream;
    extra = ds < 4 ? 0 : (ds >> 1) - 1;
    if (!br.need(extra)) return kBadStream;
    const uint32_t dist = (ds < 4 ? ds + 1u : ((2u + (ds & 1)) << extra) + 1) + br.take(extra);
    if (dist > op) return kBadStream;
    if (len > out_len - op) return kBadSize;
    t.sync();  // the literals lane 0 wrote are visible to the team
    uint8_t* dst = out + op;
    const uint8_t* src = dst - dist;
    // every source byte precedes `dst`: an overlapping copy (dist < len) repeats the last `dist` bytes
    if (dist >= len)
      for (uint32_t k = t.lane; k < len; k += t.width) dst[k] = src[k];
    else
      for (uint32_t k = t.lane; k < len; k += t.width) dst[k] = src[k % dist];
    t.sync();
    op += len;
  }
}

// Inflates the raw deflate stream [in, in + in_len) into exactly out_len bytes at out.
SAI_HD int inflate_block(const uint8_t* in, uint32_t in_len, uint8_t* out, uint32_t out_len, Tables& T, const Team& t) {
  BitReader br{in, in_len, 0, 0, 0};
  uint32_t op = 0;
  uint32_t last = 0;
  while (!last) {
    if (!br.need(3)) return kBadStream;
    last = br.take(1);
    const uint32_t type = br.take(2);
    if (type == 0) {  // stored: byte aligned LEN, NLEN, LEN bytes
      br.take(br.cnt & 7);
      br.pos -= (uint32_t)(br.cnt >> 3);  // whole bytes read ahead go back to the input
      br.buf = 0;
      br.cnt = 0;
      if (in_len - br.pos < 4) return kBadStream;
      const uint32_t len = in[br.pos] | ((uint32_t)in[br.pos + 1] << 8);
      const uint32_t nlen = in[br.pos + 2] | ((uint32_t)in[br.pos + 3] << 8);
      br.pos += 4;
      if (len != (~nlen & 0xffffu)) return kBadStream;
      if (len > in_len - br.pos) return kBadStream;
      if (len > out_len - op) return kBadSize;
      for (uint32_t k = t.lane; k < len; k += t.width) out[op + k] = in[br.pos + k];
      t.sync();
      br.pos += len;
      op += len;
    } else if (type == 1) {  // fixed Huffman codes (RFC 1951 3.2.6)
      for (int s = t.lane; s < 288; s += t.width) T.lens[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
      for (int s = t.lane; s < 30; s += t.width) T.lens[288 + s] = 5;
      t.sync();
      if (!build(T.lit, T.lens, 288, t) || !build(T.dist, T.lens + 288, 30, t)) return kBadStream;
      if (int rc = codes(T, br, out, out_len, op, t)) return rc;
    } else if (type == 2) {  // dynamic Huffman codes (RFC 1951 3.2.7)
      if (!br.need(14)) return kBadStream;
      const int nlen = (int)br.take(5) + 257, ndist = (int)br.take(5) + 1, ncode = (int)br.take(4) + 4;
      if (nlen > 286 || ndist > 30) return kBadStream;
      // the order in which the code-length code lengths are sent
      const char* order = "\x10\x11\x12\x00\x08\x07\x09\x06\x0a\x05\x0b\x04\x0c\x03\x0d\x02\x0e\x01\x0f";
      uint8_t* cl = T.lens + 300;  // the 19 code-length code lengths, out of the way of lens[0, 316)
      for (int k = 0; k < 19; ++k) {
        uint32_t v = 0;
        if (k < ncode) {
          if (!br.need(3)) return kBadStream;
          v = br.take(3);
        }
        if (t.lane == 0) cl[order[k]] = (uint8_t)v;
      }
      t.sync();
      if (!build(T.lit, cl, 19, t)) return kBadStream;
      int idx = 0;
      while (idx < nlen + ndist) {
        const int sym = decode(T.lit, br);
        if (sym < 0) return kBadStream;
        if (sym < 16) {
          if (t.lane == 0) T.lens[idx] = (uint8_t)sym;
          ++idx;
          continue;
        }
        uint32_t v = 0, rep;
        if (sym == 16) {
          if (idx == 0 || !br.need(2)) return kBadStream;
          t.sync();
          v = T.lens[idx - 1];
          rep = 3 + br.take(2);
        } else if (sym == 17) {
          if (!br.need(3)) return kBadStream;
          rep = 3 + br.take(3);
        } else {
          if (!br.need(7)) return kBadStream;
          rep = 11 + br.take(7);
        }
        if (idx + (int)rep > nlen + ndist) return kBadStream;
        if (t.lane == 0)
          for (uint32_t k = 0; k < rep; ++k) T.lens[idx + k] = (uint8_t)v;
        idx += (int)rep;
      }
      t.sync();
      if (T.lens[256] == 0) return kBadStream;  // no end-of-block code
      if (!build(T.lit, T.lens, nlen, t) || !build(T.dist, T.lens + nlen, ndist, t)) return kBadStream;
      if (int rc = codes(T, br, out, out_len, op, t)) return rc;
    } else {
      return kBadStream;
    }
  }
  return op == out_len ? kOk : kBadSize;
}

SAI_HD uint32_t min_u32(uint32_t a, uint32_t b) { return a < b ? a : b; }

// ---- CRC-32 (zlib's: reflected polynomial 0xEDB88320, initial and final complement) ----------

SAI_HD uint32_t crc_table_entry(uint32_t i) {
  for (int k = 0; k < 8; ++k) i = i & 1 ? (i >> 1) ^ 0xEDB88320u : i >> 1;
  return i;
}

// a * b modulo the CRC polynomial (bit 31 = x^0)
SAI_HD uint32_t mulmod(uint32_t a, uint32_t b) {
  uint32_t p = 0;
  for (int k = 0; k < 32; ++k) {
    if (a & (0x80000000u >> k)) p ^= b;
    b = b & 1 ? (b >> 1) ^ 0xEDB88320u : b >> 1;
  }
  return p;
}

// x^(8 n) modulo the CRC polynomial: what n zero bytes do to a CRC register
SAI_HD uint32_t x8n(uint64_t n) {
  uint32_t p = 0x80000000u, sq = 0x00800000u;  // x^0, x^8
  for (; n; n >>= 1) {
    if (n & 1) p = mulmod(sq, p);
    sq = mulmod(sq, sq);
  }
  return p;
}

// The team's share of the CRC-32 of [p, p + n): lane i takes one of `width` equal parts and returns
// its register (from 0) shifted by the bytes that follow the part; the XOR of all shares, `s`,
// gives crc32 = ~(s ^ x8n(n) * 0xFFFFFFFF).  A single lane gets the whole CRC-32 from crc_finish.
SAI_HD uint32_t crc_share(const uint8_t* p, uint32_t n, const uint32_t* table, const Team& t) {
  const uint32_t part = (n + t.width - 1) / t.width;
  const uint32_t a = min_u32(n, (uint32_t)t.lane * part), b = min_u32(n, a + part);
  uint32_t c = 0;
  for (uint32_t i = a; i < b; ++i) c = table[(c ^ p[i]) & 0xff] ^ (c >> 8);
  return c ? mulmod(x8n(n - b), c) : 0;
}
SAI_HD uint32_t crc_finish(uint32_t shares, uint32_t n) { return ~(shares ^ mulmod(x8n(n), 0xFFFFFFFFu)); }

}  // namespace infl
}  // namespace sai
