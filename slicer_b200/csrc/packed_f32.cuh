// packed_f32.cuh — two IEEE float operations in one instruction: PTX fma / add / sub / mul .rn.f32x2, which ptxas turns into
// FFMA2 / FADD2 / FMUL2 on sm_100a.  Each lane rounds to nearest even exactly like the scalar __fmaf_rn / __fadd_rn / __fsub_rn /
// __fmul_rn (no .ftz: denormal operands and results are kept), so a pair of independent scalar chains can be issued as one packed
// chain without changing a bit (slicer_selftest_packed compares them lane by lane).  A scalar operand that is the same for both
// lanes is passed as make_float2(c, c): ptxas encodes it as a broadcast register, and |x| of a lane as an operand modifier.
#pragma once
#include <cuda_runtime.h>

__device__ __forceinline__ float2 fma2_rn(float2 a, float2 b, float2 c)
{
  float2 d;
  asm("{\n.reg .b64 a, b, c, d;\n"
      "mov.b64 a, {%2, %3};\nmov.b64 b, {%4, %5};\nmov.b64 c, {%6, %7};\n"
      "fma.rn.f32x2 d, a, b, c;\n"
      "mov.b64 {%0, %1}, d;\n}"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
  return d;
}

__device__ __forceinline__ float2 add2_rn(float2 a, float2 b)
{
  float2 d;
  asm("{\n.reg .b64 a, b, d;\n"
      "mov.b64 a, {%2, %3};\nmov.b64 b, {%4, %5};\n"
      "add.rn.f32x2 d, a, b;\n"
      "mov.b64 {%0, %1}, d;\n}"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return d;
}

__device__ __forceinline__ float2 sub2_rn(float2 a, float2 b)
{
  float2 d;
  asm("{\n.reg .b64 a, b, d;\n"
      "mov.b64 a, {%2, %3};\nmov.b64 b, {%4, %5};\n"
      "sub.rn.f32x2 d, a, b;\n"
      "mov.b64 {%0, %1}, d;\n}"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return d;
}

__device__ __forceinline__ float2 mul2_rn(float2 a, float2 b)
{
  float2 d;
  asm("{\n.reg .b64 a, b, d;\n"
      "mov.b64 a, {%2, %3};\nmov.b64 b, {%4, %5};\n"
      "mul.rn.f32x2 d, a, b;\n"
      "mov.b64 {%0, %1}, d;\n}"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return d;
}

__device__ __forceinline__ float2 splat2(float c) { return make_float2(c, c); }
