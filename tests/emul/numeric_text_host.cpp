// numeric_text_host.cpp — TEST INFRASTRUCTURE ONLY.
// Compiles the device numeric formatter (etl_b200/csrc/numeric_text.cuh, the source nvcc compiles for sm_100a) for the
// host so that tests/test_numeric_text_on_host.py can compare it with a restatement of PgNumeric::to_string() on many
// spellings.  Nothing outside tests/ loads it.
#include <stdint.h>
#include <string.h>

#define __device__
#define __host__

#include "numeric_text.cuh"

// entry = the heap bytes of one numeric cell (etl_numeric_hdr + n_digits int16 digits).  The text is written by
// n_writers writers taking turns from the last to the first, as the lanes of a warp would, into a buffer pre-filled
// with 0xFF (the caller checks no such byte is left).  Returns the length, or -1 if it exceeds cap.
extern "C" int64_t emu_numeric_text(const uint8_t* entry, uint32_t n_digits, uint32_t n_writers, uint8_t* out, uint64_t cap) {
  etl_numeric_hdr h;
  memcpy(&h, entry, sizeof h);
  const int16_t* digits = reinterpret_cast<const int16_t*>(entry + sizeof h);
  const uint32_t len = etl::numeric_text_len(h, n_digits, digits);
  if (len > cap) return -1;
  memset(out, 0xFF, len);
  for (uint32_t w = n_writers; w-- > 0;) etl::numeric_text_write(h, n_digits, digits, out, w, n_writers);
  return len;
}
