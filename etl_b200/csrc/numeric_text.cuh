// numeric_text.cuh — PgNumeric::to_string() (crates/etl/src/conversions/numeric.rs:502-590: the Display arms for
// NaN / ±Infinity and format_numeric_value) over the decoder's numeric heap entry (etl_numeric_hdr + base-10000
// digits).  Plain C++ with __host__ __device__ qualifiers only, so that tests/emul/numeric_text_host.cpp can compile
// exactly this source for the host and compare it with a restatement of the reference.
//
// The text of a finite value with digits is
//   ['-'] int ['.' frac]      int  = "0" when weight < 0, else group 0 without its leading zeros ("0" if it is 0)
//                                    followed by groups 1..weight as four digits each (groups past the end are 0000)
//                                frac = scale digits: groups weight+1, weight+2, … as four digits each, the last one cut
// so every group but the first and the last fraction group has four fixed output positions, and a value can be written
// by several writers at once, writer l of n taking groups l, l+n, … (numeric_text_write).
#pragma once
#include <stdint.h>

#include "etl_decode.h"

namespace etl {

__host__ __device__ inline uint32_t numeric_group(const int16_t* digits, uint32_t n_digits, int32_t d) {
  return (d >= 0 && (uint32_t)d < n_digits) ? (uint32_t)(uint16_t)digits[d] : 0u;
}
// characters of group 0 once its leading zeros are trimmed ("0" for 0)
__host__ __device__ inline uint32_t numeric_lead_len(uint32_t g) { return g >= 1000u ? 4u : g >= 100u ? 3u : g >= 10u ? 2u : 1u; }

// Length of the text.  O(1): reads the header and at most the first digit group.
__host__ __device__ inline uint32_t numeric_text_len(const etl_numeric_hdr& h, uint32_t n_digits, const int16_t* digits) {
  if (h.kind == 1) return 3;    // NaN
  if (h.kind == 2) return 8;    // Infinity
  if (h.kind == 3) return 9;    // -Infinity
  if (n_digits == 0) return 1;  // "0", whatever the scale
  uint32_t len = h.sign ? 1u : 0u;
  len += h.weight < 0 ? 1u : numeric_lead_len(numeric_group(digits, n_digits, 0)) + 4u * (uint32_t)h.weight;
  if (h.scale) len += 1u + h.scale;
  return len;
}

// the first n characters of the k-digit decimal spelling of g (k = 4: a whole group; k = numeric_lead_len: group 0)
__host__ __device__ inline void numeric_put(uint8_t* dst, uint32_t g, uint32_t k, uint32_t n) {
  uint32_t div = k == 4u ? 1000u : k == 3u ? 100u : k == 2u ? 10u : 1u;
  for (uint32_t i = 0; i < n; i++, div /= 10u) dst[i] = (uint8_t)('0' + g / div % 10u);
}

// Writes the part of the text that belongs to writer `w` of `n_w` (w = 0, n_w = 1: all of it) at dst, which holds
// numeric_text_len bytes.  Writer 0 also writes the sign, a leading "0" and the decimal point.
__host__ __device__ inline void numeric_text_write(const etl_numeric_hdr& h, uint32_t n_digits, const int16_t* digits, uint8_t* dst,
                                                   uint32_t w, uint32_t n_w) {
  if (h.kind != 0 || n_digits == 0) {
    if (w != 0) return;
    const char* s = h.kind == 1 ? "NaN" : h.kind == 2 ? "Infinity" : h.kind == 3 ? "-Infinity" : "0";
    for (uint32_t i = 0; s[i]; i++) dst[i] = (uint8_t)s[i];
    return;
  }
  const uint32_t p0 = h.sign ? 1u : 0u;
  const int32_t weight = h.weight;
  const uint32_t n_int = weight >= 0 ? (uint32_t)weight + 1u : 0u;       // integer groups
  const uint32_t lead = weight >= 0 ? numeric_lead_len(numeric_group(digits, n_digits, 0)) : 1u;
  const uint32_t frac0 = p0 + lead + (n_int ? 4u * (n_int - 1u) : 0u) + 1u; // first fraction digit
  const uint32_t n_frac = (h.scale + 3u) / 4u;                             // fraction groups
  if (w == 0) {
    if (h.sign) dst[0] = '-';
    if (weight < 0) dst[p0] = '0';
    if (h.scale) dst[frac0 - 1] = '.';
  }
  for (uint32_t t = w; t < n_int + n_frac; t += n_w) {
    if (t < n_int) {
      const uint32_t g = numeric_group(digits, n_digits, (int32_t)t);
      if (t == 0) numeric_put(dst + p0, g, lead, lead);
      else numeric_put(dst + p0 + lead + 4u * (t - 1u), g, 4, 4);
    } else {
      const uint32_t j = t - n_int;
      const uint32_t left = h.scale - 4u * j;
      numeric_put(dst + frac0 + 4u * j, numeric_group(digits, n_digits, weight + 1 + (int32_t)j), 4, left < 4u ? left : 4u);
    }
  }
}

}  // namespace etl
