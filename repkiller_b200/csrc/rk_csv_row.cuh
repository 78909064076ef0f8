// The rules of one GECKO CSV row, shared by the host parser (readFragment, below; host/FragmentsDatabase.cpp) and the
// device parser (k9_csv.cu).  atoll / strtof are what the reference calls; the two helpers below return the same values
// for the plain tokens a GECKO file is made of (all digits; digits[.digits]) without the copy, the locale machinery and
// the errno round trip, and say "no" for everything else (signs, blanks, exponents, overlong tokens), which then takes
// the library call.  Compiled by nvcc they are __host__ __device__: the device decides a row only where these say yes,
// so both sides run the same code on the same tokens (IEEE round-to-nearest division and narrowing on both).
#pragma once

#include <cstddef>
#include <cstdint>
#include <cstring>

#if defined(__CUDACC__)
#define RK_CSV_HD __host__ __device__
#else
#define RK_CSV_HD
#endif

namespace rk_csv {

#define RK_CSV_P10 {1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11, 1e12, 1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19, 1e20, 1e21, 1e22}
#if defined(__CUDACC__)
__constant__ double P10_dev[23] = RK_CSV_P10;
#endif

RK_CSV_HD inline double p10(int k) {  // 10^k, k <= 22: every one an exact double
#if defined(__CUDA_ARCH__)
  return P10_dev[k];
#else
  static const double P10[23] = RK_CSV_P10;
  return P10[k];
#endif
}
#undef RK_CSV_P10

RK_CSV_HD inline bool plain_u64(const char *p, size_t n, uint64_t &v) {  // 1..18 digits: below 2^63, atoll returns the same
  if (n == 0 || n > 18) return false;
  uint64_t x = 0;
  for (size_t i = 0; i < n; ++i) {
    const unsigned c = (unsigned char)p[i] - '0';
    if (c > 9) return false;
    x = x * 10 + c;
  }
  v = x;
  return true;
}

// digits[.digits] with an integer mantissa below 2^53 and at most 22 fraction digits: mantissa and power of ten are
// exact doubles, their quotient is the correctly rounded double, and narrowing it gives the correctly rounded float
// (what strtof returns) unless the double sits on the midpoint of two floats — then the library decides.
RK_CSV_HD inline bool plain_float(const char *p, size_t n, float &out) {
  uint64_t m = 0;
  int digits = 0, frac = 0;
  bool dot = false;
  for (size_t i = 0; i < n; ++i) {
    const unsigned c = (unsigned char)p[i] - '0';
    if (c <= 9) {
      if (++digits > 18) return false;
      m = m * 10 + c;
      frac += dot;
    } else if (p[i] == '.' && !dot) {
      dot = true;
    } else {
      return false;
    }
  }
  if (digits == 0 || frac > 22 || m >= (1ull << 53)) return false;
  const double d = (double)m / p10(frac);
  uint64_t bits;
#if defined(__CUDA_ARCH__)
  bits = (uint64_t)__double_as_longlong(d);
#else
  memcpy(&bits, &d, sizeof bits);
#endif
  const uint32_t low = (uint32_t)(bits & 0x1FFFFFFFu);  // the 29 bits a float drops
  if (low >= 0x0FFFFFFFu && low <= 0x10000001u) return false;
  out = (float)d;
  return true;
}

}  // namespace rk_csv

#if !defined(__CUDA_ARCH__)  // host code (the host pass of nvcc included)
#include <cerrno>
#include <cstdlib>

#include "host/structs.h"

// One CSV row -> record.  Semantics of the reference's readFragment (FragmentsDatabase.cpp:17-50), which
// tokenises with 14 x getline(stream, buf, ','):
//  * a token ends at ',' or at the end of the row; an EMPTY token rejects the row (:25);
//  * once the row is exhausted the extraction fails and buf keeps the previous token, so a short row is
//    padded with its last field ("Frag,5" loads with every numeric field 5 and strand '5');
//  * a trailing ',' produces one empty token (row rejected);
//  * field 0 must be "Frag" (:29); numeric fields through atoll; similarity AND ident from stof(field 10)
//    (:39-40; field 9 is ignored); a row whose similarity does not parse is rejected (:46-48).
// Host only: the device parser (k9_csv.cu) applies the same token rules and leaves every row these helpers do not
// decide to this function.
inline bool readFragment(FragFile *frag, const char *line, size_t len) {
  using rk_csv::plain_float;
  using rk_csv::plain_u64;
  const char *tok[14];
  size_t tlen[14];
  size_t pos = 0;
  bool exhausted = false;
  const char *cur = nullptr;
  size_t curlen = 0;
  for (int i = 0; i < 14; ++i) {
    if (!exhausted) {
      const size_t s = pos;
      while (pos < len && line[pos] != ',') ++pos;
      cur = line + s;
      curlen = pos - s;
      if (pos < len) ++pos;
      else exhausted = true;
    }
    if (curlen == 0) return false;
    tok[i] = cur;
    tlen[i] = curlen;
  }
  if (!(tlen[0] == 4 && memcmp(tok[0], "Frag", 4) == 0)) return false;
  char buf[72];
  auto cstr = [&](int i) -> const char * {
    const size_t l = tlen[i] < 71 ? tlen[i] : 71;
    memcpy(buf, tok[i], l);
    buf[l] = 0;
    return buf;
  };
  auto num = [&](int i) -> long long {
    uint64_t v;
    return plain_u64(tok[i], tlen[i], v) ? (long long)v : atoll(cstr(i));
  };
  frag->xStart = (uint64_t)num(1);
  frag->yStart = (uint64_t)num(2);
  frag->diag = (int64_t)frag->xStart - (int64_t)frag->yStart;
  frag->xEnd = (uint64_t)num(3);
  frag->yEnd = (uint64_t)num(4);
  frag->strand = tok[5][0];
  frag->block = num(6);
  frag->length = (uint64_t)num(7);
  frag->score = (uint64_t)num(8);
  float sim;
  if (!plain_float(tok[10], tlen[10], sim)) {
    const char *s = cstr(10);
    char *endp = nullptr;
    errno = 0;
    sim = strtof(s, &endp);  // std::stof: invalid_argument when nothing converts, out_of_range on ERANGE
    if (endp == s || errno == ERANGE) return false;
  }
  frag->ident = (uint64_t)sim;
  frag->similarity = sim;
  frag->seqX = 0;
  frag->seqY = 1;
  memset(frag->evalue, 0, sizeof frag->evalue);
  return true;
}
#endif
