// Cells of a score file read the way pandas' C parser reads them with the reference's
// read_csv(sep="\t", na_values=["nan"], index_col=False) (sai/sai.py:175), for the device outlier
// tables (table_kernels.cu) and its host build (tests).
//
// xstrtod is pandas' precise_xstrtod (pandas/_libs/src/parser/tokenizer.c), the converter of
// float_precision=None: at most 17 digits accumulated as number * 10 + d, the rest move the
// exponent, then one multiplication or division by a double power of ten.  It does not round
// correctly (the reference's own tables show its last digits), so a device path that parsed
// correctly would print different text.  All arithmetic is plain IEEE double; the library is built
// with --fmad=false, so the device gives the host's bits.
//
// classify_cell sorts a cell into the classes pandas' type inference distinguishes, conservatively:
// kUnsure marks every spelling whose dtype or value this code does not reproduce (whitespace, '+',
// bool and infinity spellings other than "inf" / "-inf", int64 overflow, bytes outside printable
// ASCII), and the caller reads such a file on the host.
//
// __host__ __device__ under nvcc; the same header compiles as plain C++.
#pragma once
#include <stdint.h>

#include "format_double.cuh"

namespace sai {
namespace parse {

// kBigInt / kNegZero mark integers pandas reads differently as int64 cast to float64 and with its
// float parser: beyond 2^53 or written with more than 17 digits (leading zeros count: the parser
// keeps the first 17 digits only), and "-0" (0.0 or -0.0)
enum : uint8_t { kInt = 1, kFloat = 2, kNa = 4, kText = 8, kUnsure = 16, kBigInt = 32, kNegZero = 64 };

#define SAI_PARSE_POW10_TABLE { \
  1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11, 1e12, 1e13, 1e14, 1e15, 1e16, 1e17, \
  1e18, 1e19, 1e20, 1e21, 1e22, 1e23, 1e24, 1e25, 1e26, 1e27, 1e28, 1e29, 1e30, 1e31, 1e32, 1e33, \
  1e34, 1e35, 1e36, 1e37, 1e38, 1e39, 1e40, 1e41, 1e42, 1e43, 1e44, 1e45, 1e46, 1e47, 1e48, 1e49, \
  1e50, 1e51, 1e52, 1e53, 1e54, 1e55, 1e56, 1e57, 1e58, 1e59, 1e60, 1e61, 1e62, 1e63, 1e64, 1e65, \
  1e66, 1e67, 1e68, 1e69, 1e70, 1e71, 1e72, 1e73, 1e74, 1e75, 1e76, 1e77, 1e78, 1e79, 1e80, 1e81, \
  1e82, 1e83, 1e84, 1e85, 1e86, 1e87, 1e88, 1e89, 1e90, 1e91, 1e92, 1e93, 1e94, 1e95, 1e96, 1e97, \
  1e98, 1e99, 1e100, 1e101, 1e102, 1e103, 1e104, 1e105, 1e106, 1e107, 1e108, 1e109, 1e110, 1e111, \
  1e112, 1e113, 1e114, 1e115, 1e116, 1e117, 1e118, 1e119, 1e120, 1e121, 1e122, 1e123, 1e124, 1e125, \
  1e126, 1e127, 1e128, 1e129, 1e130, 1e131, 1e132, 1e133, 1e134, 1e135, 1e136, 1e137, 1e138, 1e139, \
  1e140, 1e141, 1e142, 1e143, 1e144, 1e145, 1e146, 1e147, 1e148, 1e149, 1e150, 1e151, 1e152, 1e153, \
  1e154, 1e155, 1e156, 1e157, 1e158, 1e159, 1e160, 1e161, 1e162, 1e163, 1e164, 1e165, 1e166, 1e167, \
  1e168, 1e169, 1e170, 1e171, 1e172, 1e173, 1e174, 1e175, 1e176, 1e177, 1e178, 1e179, 1e180, 1e181, \
  1e182, 1e183, 1e184, 1e185, 1e186, 1e187, 1e188, 1e189, 1e190, 1e191, 1e192, 1e193, 1e194, 1e195, \
  1e196, 1e197, 1e198, 1e199, 1e200, 1e201, 1e202, 1e203, 1e204, 1e205, 1e206, 1e207, 1e208, 1e209, \
  1e210, 1e211, 1e212, 1e213, 1e214, 1e215, 1e216, 1e217, 1e218, 1e219, 1e220, 1e221, 1e222, 1e223, \
  1e224, 1e225, 1e226, 1e227, 1e228, 1e229, 1e230, 1e231, 1e232, 1e233, 1e234, 1e235, 1e236, 1e237, \
  1e238, 1e239, 1e240, 1e241, 1e242, 1e243, 1e244, 1e245, 1e246, 1e247, 1e248, 1e249, 1e250, 1e251, \
  1e252, 1e253, 1e254, 1e255, 1e256, 1e257, 1e258, 1e259, 1e260, 1e261, 1e262, 1e263, 1e264, 1e265, \
  1e266, 1e267, 1e268, 1e269, 1e270, 1e271, 1e272, 1e273, 1e274, 1e275, 1e276, 1e277, 1e278, 1e279, \
  1e280, 1e281, 1e282, 1e283, 1e284, 1e285, 1e286, 1e287, 1e288, 1e289, 1e290, 1e291, 1e292, 1e293, \
  1e294, 1e295, 1e296, 1e297, 1e298, 1e299, 1e300, 1e301, 1e302, 1e303, 1e304, 1e305, 1e306, 1e307, \
  1e308}
#ifdef __CUDACC__
static __device__ const double kPow10Dev[309] = SAI_PARSE_POW10_TABLE;
#endif
static const double kPow10Host[309] = SAI_PARSE_POW10_TABLE;

SAI_FMT_HD double pow10(int i) {
#ifdef __CUDA_ARCH__
  return kPow10Dev[i];
#else
  return kPow10Host[i];
#endif
}

SAI_FMT_HD bool is_digit(char c) { return c >= '0' && c <= '9'; }
SAI_FMT_HD bool is_space(char c) { return c == ' ' || (c >= '\t' && c <= '\r'); }

// precise_xstrtod over s[0, n): *out is its result; true when pandas accepts the cell as a float
// (no range error and the whole cell consumed)
SAI_FMT_HD bool xstrtod(const char* s, int n, double* out) {
  int i = 0;
  while (i < n && is_space(s[i])) ++i;
  bool neg = false;
  if (i < n && (s[i] == '-' || s[i] == '+')) neg = s[i++] == '-';
  double number = 0.;
  int exponent = 0, num_digits = 0, num_decimals = 0;
  for (; i < n && is_digit(s[i]); ++i) {
    if (num_digits < 17) {
      number = number * 10. + (s[i] - '0');
      ++num_digits;
    } else {
      ++exponent;
    }
  }
  if (i < n && s[i] == '.') {
    ++i;
    for (; num_digits < 17 && i < n && is_digit(s[i]); ++i) {
      number = number * 10. + (s[i] - '0');
      ++num_digits;
      ++num_decimals;
    }
    if (num_digits >= 17)
      while (i < n && is_digit(s[i])) ++i;
    exponent -= num_decimals;
  }
  if (num_digits == 0) {
    *out = 0.;
    return false;
  }
  if (neg) number = -number;
  if (i < n && (s[i] == 'e' || s[i] == 'E')) {
    int j = i + 1;
    bool eneg = false;
    if (j < n && (s[j] == '-' || s[j] == '+')) eneg = s[j++] == '-';
    int nd = 0;
    uint32_t e = 0;  // pandas accumulates up to 17 digits in an int; wraps the same way
    for (; nd < 17 && j < n && is_digit(s[j]); ++j, ++nd) e = e * 10u + (uint32_t)(s[j] - '0');
    exponent = (int)((uint32_t)exponent + (eneg ? 0u - e : e));
    i = nd ? j : j - 1;  // no exponent digits: the 'e' (or its sign) is not consumed
  }
  bool range = false;
  if (exponent > 308) {
    number = __builtin_huge_val();
    range = true;
  } else if (exponent > 0) {
    number *= pow10(exponent);
  } else if (exponent < -308) {
    if (exponent < -616) {
      number = 0.;
    } else {
      number /= pow10(-308 - exponent);
      number /= pow10(308);
    }
  } else {
    number /= pow10(-exponent);
  }
  if (number == __builtin_huge_val() || number == -__builtin_huge_val()) range = true;
  while (i < n && is_space(s[i])) ++i;
  *out = number;
  return !range && i == n;
}

SAI_FMT_HD bool equals(const char* s, int n, const char* lit) {
  int i = 0;
  for (; i < n; ++i)
    if (lit[i] != s[i]) return false;
  return lit[i] == 0;
}

// pandas' STR_NA_VALUES plus "nan" (na_values=["nan"] with keep_default_na)
SAI_FMT_HD bool is_na(const char* s, int n) {
  if (n == 0) return true;
  if (n > 9) return false;
  const char* na[] = {"#N/A", "#N/A N/A", "#NA", "-1.#IND", "-1.#QNAN", "-NaN", "-nan", "1.#IND", "1.#QNAN",
                      "<NA>", "N/A", "NA", "NULL", "NaN", "None", "n/a", "nan", "null"};
  for (const char* w : na)
    if (equals(s, n, w)) return true;
  return false;
}

// words pandas may read as a float, a bool or NA in some spelling (compared in lower case, after
// one optional sign)
SAI_FMT_HD bool is_special_word(const char* s, int n) {
  if (n > 0 && (s[0] == '+' || s[0] == '-')) ++s, --n;
  if (n > 9) return false;
  char low[9];
  for (int i = 0; i < n; ++i) low[i] = (s[i] >= 'A' && s[i] <= 'Z') ? (char)(s[i] + 32) : s[i];
  const char* words[] = {"inf", "infinity", "nan", "true", "false", "null", "none", "na", "n/a",
                         "<na>", "#na", "#n/a", "1.#inf", "1.#ind", "1.#qnan", "nat"};
  for (const char* w : words)
    if (equals(low, n, w)) return true;
  return false;
}

// [-]?[0-9]+ into *v; false on int64 overflow or any other spelling
SAI_FMT_HD bool parse_int64(const char* s, int n, int64_t* v) {
  int i = 0;
  const bool neg = n > 0 && s[0] == '-';
  if (neg) ++i;
  if (i == n) return false;
  uint64_t m = 0;
  const uint64_t lim = neg ? 9223372036854775808ull : 9223372036854775807ull;
  for (; i < n; ++i) {
    if (!is_digit(s[i])) return false;
    const uint64_t d = (uint64_t)(s[i] - '0');
    if (m > (lim - d) / 10) return false;
    m = m * 10 + d;
  }
  *v = neg ? (int64_t)(0 - m) : (int64_t)m;
  return true;
}

// -?digits*(.digits*)?([eE][+-]?digits{1,4})? with at least one mantissa digit
SAI_FMT_HD bool float_grammar(const char* s, int n) {
  int i = 0, digits = 0;
  if (i < n && s[i] == '-') ++i;
  for (; i < n && is_digit(s[i]); ++i) ++digits;
  if (i < n && s[i] == '.')
    for (++i; i < n && is_digit(s[i]); ++i) ++digits;
  if (digits == 0) return false;
  if (i < n && (s[i] == 'e' || s[i] == 'E')) {
    ++i;
    if (i < n && (s[i] == '-' || s[i] == '+')) ++i;
    int ed = 0;
    for (; i < n && is_digit(s[i]); ++i) ++ed;
    if (ed < 1 || ed > 4) return false;
  }
  return i == n;
}

// the value of a cell of class kFloat: "inf" / "-inf" or what xstrtod reads
SAI_FMT_HD double float_cell(const char* s, int n) {
  if (equals(s, n, "inf")) return __builtin_huge_val();
  if (equals(s, n, "-inf")) return -__builtin_huge_val();
  double v;
  xstrtod(s, n, &v);
  return v;
}

SAI_FMT_HD uint8_t classify_cell(const char* s, int n) {
  bool numeric_chars = true;
  for (int i = 0; i < n; ++i) {
    const char c = s[i];
    if (c < 0x21 || c > 0x7e) return kUnsure;
    numeric_chars &= is_digit(c) || c == '.' || c == 'e' || c == 'E' || c == '+' || c == '-';
  }
  if (is_na(s, n)) return kNa;
  if (equals(s, n, "inf") || equals(s, n, "-inf")) return kFloat;
  if (is_special_word(s, n)) return kUnsure;
  if (!numeric_chars) return kText;
  int64_t v;
  bool all_int = n > 0;
  for (int i = (n > 0 && s[0] == '-') ? 1 : 0; i < n; ++i) all_int &= is_digit(s[i]);
  if (all_int && !(n == 1 && s[0] == '-')) {
    if (!parse_int64(s, n, &v)) return kUnsure;
    const uint64_t a = v < 0 ? 0 - (uint64_t)v : (uint64_t)v;
    const int digits = s[0] == '-' ? n - 1 : n;
    if (a > (1ull << 53) || digits > 17) return kInt | kBigInt;
    return (v == 0 && s[0] == '-') ? kInt | kNegZero : kInt;
  }
  double d;
  if (float_grammar(s, n) && xstrtod(s, n, &d)) return kFloat;
  return kUnsure;
}

}  // namespace parse
}  // namespace sai
