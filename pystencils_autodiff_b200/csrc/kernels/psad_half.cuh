// psad_half.cuh — float16 fields: IEEE binary16 storage, fp32 (or fp64) arithmetic.  Included after psad_common.cuh by
// the kernels that have float16 fields only.  Values stay raw 16-bit words in memory and are converted with inline PTX
// (no cuda_fp16.h: the NVRTC-compiled kernels include no system headers, see psad_args.h): cvt.f32.f16 where a value
// enters the registers, cvt.rn.f16x2.f32 (two cells per instruction) where a result is stored — one rounding per cell.
#ifndef PSAD_HALF_CUH
#define PSAD_HALF_CUH

PSAD_DEV float psad_h2f(unsigned short h) {
  float f;
  asm("cvt.f32.f16 %0, %1;" : "=f"(f) : "h"(h));
  return f;
}
PSAD_DEV unsigned short psad_f2h(float f) {
  unsigned short h;
  asm("cvt.rn.f16.f32 %0, %1;" : "=h"(h) : "f"(f));
  return h;
}
PSAD_DEV unsigned short psad_d2h(double d) {   // one rounding from fp64 (data_type='double'), not two through fp32
  unsigned short h;
  asm("cvt.rn.f16.f64 %0, %1;" : "=h"(h) : "d"(d));
  return h;
}
// two floats -> one 32-bit word of two halves (lo in the low 16 bits: the lower address)
PSAD_DEV psad_u32 psad_f2h2(float lo, float hi) {
  psad_u32 r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
PSAD_DEV psad_u32 psad_d2h2(double lo, double hi) { return (psad_u32)psad_d2h(lo) | ((psad_u32)psad_d2h(hi) << 16); }
// one 32-bit word of two halves -> two floats
PSAD_DEV void psad_h22f(psad_u32 w, float& lo, float& hi) {
  asm("{\n.reg .f16 l, h;\nmov.b32 {l, h}, %2;\ncvt.f32.f16 %0, l;\ncvt.f32.f16 %1, h;\n}" : "=f"(lo), "=f"(hi) : "r"(w));
}

// A float16 element in memory.  Reads convert to float, writes round from float / double: the generic kernel's
// `(CT)p[i]` and `p[i] = (T)v` work on it unchanged.
struct psad_half {
  unsigned short bits;
  psad_half() = default;
  PSAD_DEV psad_half(float f) : bits(psad_f2h(f)) {}
  PSAD_DEV psad_half(double d) : bits(psad_d2h(d)) {}
  PSAD_DEV operator float() const { return psad_h2f(bits); }
};

// shared -> registers: four halves (one aligned 8-byte LDS.64) into four floats of the register window
PSAD_DEV void psad_lds_h4(const psad_half* p, float* e) {
  const uint2 v = *reinterpret_cast<const uint2*>(p);
  psad_h22f(v.x, e[0], e[1]);
  psad_h22f(v.y, e[2], e[3]);
}
// registers -> global: four results rounded to halves, one aligned 8-byte store (cache policy as psad_stg_vec)
PSAD_DEV void psad_stg_h4_bits(psad_half* p, uint2 v) {
#if PSAD_STORE_MODE == 0
  *reinterpret_cast<uint2*>(p) = v;
#elif PSAD_STORE_MODE == 2
  __stwt(reinterpret_cast<uint2*>(p), v);
#else
  __stcs(reinterpret_cast<uint2*>(p), v);
#endif
}
PSAD_DEV void psad_stg_h4(psad_half* p, const float* e) {
  psad_stg_h4_bits(p, make_uint2(psad_f2h2(e[0], e[1]), psad_f2h2(e[2], e[3])));
}
PSAD_DEV void psad_stg_h4(psad_half* p, const double* e) {
  psad_stg_h4_bits(p, make_uint2(psad_d2h2(e[0], e[1]), psad_d2h2(e[2], e[3])));
}

#endif
