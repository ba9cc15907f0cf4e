// Host stand-in for csrc/kernels/psad_half.cuh (float16 storage, fp32 / fp64 arithmetic).  TEST INFRASTRUCTURE: the
// conversions use g++'s _Float16 (IEEE binary16, round to nearest even like cvt.rn), so the replay rounds every stored
// cell exactly as the device does.  The same file is in every cpu_shim* directory.
#ifndef PSAD_HALF_CUH
#define PSAD_HALF_CUH

#include <cstring>

struct psad_half {
  unsigned short bits;
  psad_half() = default;
  psad_half(float f) { const _Float16 h = (_Float16)f; std::memcpy(&bits, &h, 2); }
  psad_half(double d) { const _Float16 h = (_Float16)d; std::memcpy(&bits, &h, 2); }
  operator float() const { _Float16 h; std::memcpy(&h, &bits, 2); return (float)h; }
};

static inline void psad_lds_h4(const psad_half* p, float* e) {
  for (int i = 0; i < 4; ++i) e[i] = (float)p[i];
}
static inline void psad_stg_h4(psad_half* p, const float* e) {
  for (int i = 0; i < 4; ++i) p[i] = psad_half(e[i]);
}
static inline void psad_stg_h4(psad_half* p, const double* e) {
  for (int i = 0; i < 4; ++i) p[i] = psad_half(e[i]);
}

#endif
