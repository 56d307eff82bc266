// Text of numbers exactly as CPython prints them, for the score-file writer (format_kernels.cu).
//
// format_double: repr(float) -- the shortest decimal string that reads back to the same double, the
// one closest to the exact value when several are equally short (Python's dtoa mode 0), laid out
// positionally when the decimal exponent e satisfies -4 <= e < 16 ("0.0001", "1234.5", "1e+16"
// otherwise, with at least two exponent digits), "nan", "inf", "-inf", "-0.0".  The digits come from
// Ryu (Adams, "Ryu: fast float-to-string conversion", PLDI 2018): the interval of decimals that round
// to the double is scaled by a 125-bit power of five (format_pow5.cuh) and digits are removed while
// both ends still differ.  str(np.float64(x)) prints the same text (tests/test_format_double.py).
//
// __host__ __device__ under nvcc; the same header compiles as plain C++.
#pragma once
#include <stdint.h>
#include <string.h>

#include "format_pow5.cuh"

#ifdef __CUDACC__
#define SAI_FMT_HD __host__ __device__ __forceinline__
#else
#define SAI_FMT_HD inline
#endif

namespace sai {
namespace fmt {

constexpr int kMaxDoubleChars = 32;  // longest is 24 ("-2.2250738585072014e-308")

#ifdef __CUDACC__
static __device__ const uint64_t kPow5Dev[SAI_FMT_POW5_COUNT][2] = SAI_FMT_POW5_TABLE;
static __device__ const uint64_t kPow5InvDev[SAI_FMT_POW5_INV_COUNT][2] = SAI_FMT_POW5_INV_TABLE;
#endif
static const uint64_t kPow5Host[SAI_FMT_POW5_COUNT][2] = SAI_FMT_POW5_TABLE;
static const uint64_t kPow5InvHost[SAI_FMT_POW5_INV_COUNT][2] = SAI_FMT_POW5_INV_TABLE;

SAI_FMT_HD const uint64_t* pow5(int i) {
#ifdef __CUDA_ARCH__
  return kPow5Dev[i];
#else
  return kPow5Host[i];
#endif
}
SAI_FMT_HD const uint64_t* pow5_inv(int i) {
#ifdef __CUDA_ARCH__
  return kPow5InvDev[i];
#else
  return kPow5InvHost[i];
#endif
}

// ceil(log2(5^e)) for e >= 1 (1 for e = 0), floor(log10(2^e)), floor(log10(5^e)); exact in range
SAI_FMT_HD int32_t pow5bits(int32_t e) { return (int32_t)(((uint32_t)e * 1217359u) >> 19) + 1; }
SAI_FMT_HD uint32_t log10pow2(int32_t e) { return ((uint32_t)e * 78913u) >> 18; }
SAI_FMT_HD uint32_t log10pow5(int32_t e) { return ((uint32_t)e * 732923u) >> 20; }

SAI_FMT_HD uint32_t pow5_factor(uint64_t v) {
  uint32_t n = 0;
  for (; v % 5 == 0; v /= 5) ++n;
  return n;
}
SAI_FMT_HD bool multiple_of_pow5(uint64_t v, uint32_t p) { return pow5_factor(v) >= p; }
SAI_FMT_HD bool multiple_of_pow2(uint64_t v, uint32_t p) { return (v & ((1ull << p) - 1)) == 0; }

// (m * mul) >> j for the 125-bit mul = {low, high}, j >= 64
SAI_FMT_HD uint64_t mul_shift(uint64_t m, const uint64_t* mul, int32_t j) {
  const unsigned __int128 b0 = (unsigned __int128)m * mul[0];
  const unsigned __int128 b2 = (unsigned __int128)m * mul[1];
  return (uint64_t)(((b0 >> 64) + b2) >> (j - 64));
}

struct Decimal {
  uint64_t digits;  // 1..17 decimal digits, no trailing zero required
  int32_t exp;      // value = digits * 10^exp
};

// Shortest decimal of a finite nonzero double given its IEEE mantissa and biased exponent.
SAI_FMT_HD Decimal shortest(uint64_t ieee_m, uint32_t ieee_e) {
  int32_t e2;
  uint64_t m2;
  if (ieee_e == 0) {
    e2 = 1 - 1023 - 52 - 2;
    m2 = ieee_m;
  } else {
    e2 = (int32_t)ieee_e - 1023 - 52 - 2;
    m2 = (1ull << 52) | ieee_m;
  }
  const bool accept_bounds = (m2 & 1) == 0;  // round-half-even reading accepts the interval's ends
  const uint64_t mv = 4 * m2;
  const uint32_t mm_shift = ieee_m != 0 || ieee_e <= 1;  // the lower neighbour is half as far at a power of two
  uint64_t vr, vp, vm;
  int32_t e10;
  bool vm_tz = false, vr_tz = false;  // the removed digits of vm / vr are all zero
  if (e2 >= 0) {
    const uint32_t q = log10pow2(e2) - (e2 > 3);
    e10 = (int32_t)q;
    const int32_t k = 125 + pow5bits((int32_t)q) - 1;
    const int32_t i = -e2 + (int32_t)q + k;
    const uint64_t* mul = pow5_inv((int)q);
    vr = mul_shift(4 * m2, mul, i);
    vp = mul_shift(4 * m2 + 2, mul, i);
    vm = mul_shift(4 * m2 - 1 - mm_shift, mul, i);
    if (q <= 21) {
      if (mv % 5 == 0) {
        vr_tz = multiple_of_pow5(mv, q);
      } else if (accept_bounds) {
        vm_tz = multiple_of_pow5(mv - 1 - mm_shift, q);
      } else {
        vp -= multiple_of_pow5(mv + 2, q);
      }
    }
  } else {
    const uint32_t q = log10pow5(-e2) - (-e2 > 1);
    e10 = (int32_t)q + e2;
    const int32_t i = -e2 - (int32_t)q;
    const int32_t k = pow5bits(i) - 125;
    const int32_t j = (int32_t)q - k;
    const uint64_t* mul = pow5(i);
    vr = mul_shift(4 * m2, mul, j);
    vp = mul_shift(4 * m2 + 2, mul, j);
    vm = mul_shift(4 * m2 - 1 - mm_shift, mul, j);
    if (q <= 1) {
      vr_tz = true;
      if (accept_bounds) {
        vm_tz = mm_shift == 1;
      } else {
        --vp;
      }
    } else if (q < 63) {
      vr_tz = multiple_of_pow2(mv, q);
    }
  }
  int32_t removed = 0;
  uint64_t out;
  if (vm_tz || vr_tz) {  // exact ends or an exact halfway digit: track the removed digits
    uint32_t last = 0;
    for (; vp / 10 > vm / 10; ++removed) {
      vm_tz &= vm % 10 == 0;
      vr_tz &= last == 0;
      last = (uint32_t)(vr % 10);
      vr /= 10;
      vp /= 10;
      vm /= 10;
    }
    if (vm_tz) {
      for (; vm % 10 == 0; ++removed) {
        vr_tz &= last == 0;
        last = (uint32_t)(vr % 10);
        vr /= 10;
        vp /= 10;
        vm /= 10;
      }
    }
    if (vr_tz && last == 5 && vr % 2 == 0) last = 4;  // exactly halfway: round to even
    out = vr + ((vr == vm && (!accept_bounds || !vm_tz)) || last >= 5);
  } else {
    bool round_up = false;
    if (vp / 100 > vm / 100) {
      round_up = vr % 100 >= 50;
      vr /= 100;
      vp /= 100;
      vm /= 100;
      removed += 2;
    }
    for (; vp / 10 > vm / 10; ++removed) {
      round_up = vr % 10 >= 5;
      vr /= 10;
      vp /= 10;
      vm /= 10;
    }
    out = vr + (vr == vm || round_up);
  }
  return Decimal{out, e10 + removed};
}

SAI_FMT_HD int decimal_length(uint64_t v) {
  int n = 1;
  for (; v >= 10; v /= 10) ++n;
  return n;
}

// digits of v right-aligned in out[0 .. n), n = decimal_length(v)
SAI_FMT_HD void put_digits(uint64_t v, char* out, int n) {
  for (int i = n - 1; i >= 0; --i) {
    out[i] = (char)('0' + v % 10);
    v /= 10;
  }
}

// str(int): returns the length (<= 20)
SAI_FMT_HD int format_int64(int64_t v, char* out) {
  int n = 0;
  uint64_t u = (uint64_t)v;
  if (v < 0) {
    out[n++] = '-';
    u = 0 - u;
  }
  const int d = decimal_length(u);
  put_digits(u, out + n, d);
  return n + d;
}

SAI_FMT_HD int int64_length(int64_t v) {
  return v < 0 ? 1 + decimal_length(0 - (uint64_t)v) : decimal_length((uint64_t)v);
}

// repr(float(x)) into out (kMaxDoubleChars bytes); returns the length
SAI_FMT_HD int format_double(double x, char* out) {
  uint64_t bits;
  memcpy(&bits, &x, sizeof bits);
  const bool neg = bits >> 63;
  const uint64_t ieee_m = bits & ((1ull << 52) - 1);
  const uint32_t ieee_e = (uint32_t)(bits >> 52) & 0x7ff;
  int n = 0;
  if (ieee_e == 0x7ff) {
    if (ieee_m) {
      memcpy(out, "nan", 3);
      return 3;
    }
    if (neg) out[n++] = '-';
    memcpy(out + n, "inf", 3);
    return n + 3;
  }
  if (neg) out[n++] = '-';
  if (ieee_e == 0 && ieee_m == 0) {
    memcpy(out + n, "0.0", 3);
    return n + 3;
  }
  const Decimal d = shortest(ieee_m, ieee_e);
  const int len = decimal_length(d.digits);
  char dig[20];
  put_digits(d.digits, dig, len);
  const int decpt = len + d.exp;  // value = 0.dig * 10^decpt
  if (decpt > -4 && decpt <= 16) {
    if (decpt <= 0) {
      out[n++] = '0';
      out[n++] = '.';
      for (int i = 0; i < -decpt; ++i) out[n++] = '0';
      for (int i = 0; i < len; ++i) out[n++] = dig[i];
    } else if (decpt < len) {
      for (int i = 0; i < decpt; ++i) out[n++] = dig[i];
      out[n++] = '.';
      for (int i = decpt; i < len; ++i) out[n++] = dig[i];
    } else {
      for (int i = 0; i < len; ++i) out[n++] = dig[i];
      for (int i = len; i < decpt; ++i) out[n++] = '0';
      out[n++] = '.';
      out[n++] = '0';
    }
    return n;
  }
  out[n++] = dig[0];
  if (len > 1) {
    out[n++] = '.';
    for (int i = 1; i < len; ++i) out[n++] = dig[i];
  }
  int e = decpt - 1;
  out[n++] = 'e';
  out[n++] = e < 0 ? '-' : '+';
  if (e < 0) e = -e;
  if (e < 10) out[n++] = '0';
  const int el = decimal_length((uint64_t)e);
  put_digits((uint64_t)e, out + n, el);
  return n + el;
}

}  // namespace fmt
}  // namespace sai
