// Operand formats of the tensor-core kernels (vlg_tc.cu, vlg_decode.cu): where each of a decoder's four GEMMs finds
// its weight image inside the packed record and its operands in a chain's 256 tensor-memory columns, and the fp16 /
// TF32 conversions that build the activation operands.  sm_100a only.
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>

#include "vlg_common.cuh"

#ifndef VLG_TC_G_AHEAD
#define VLG_TC_G_AHEAD 1               // single-term backward: next item's dE/dx rows built under the current B2
#endif

namespace vlg {
namespace {

constexpr int STAGE_BYTES = 16384;    // one weight stage of a shared-memory ring

// the four tensor-core GEMMs of one decoder
struct OpInfo {
  int img_off;   // float offset of the B image inside the decoder record
  int nstages;   // 16 KB stages
  int n;         // MMA N
  int nk;        // MMAs per stage (8 TMEM columns of A each: 8 tf32 or 16 fp16 contraction indices)
  int a_col;     // chain-relative TMEM column of A
  int d_col;     // chain-relative TMEM column of D
  int img_lo;    // 3-term mode: float offset of the residual image
};
// operand formats of the tensor-core kernel
constexpr int FMT_TF32 = 0, FMT_F16 = 1, FMT_F16X3 = 2, FMT_F16X3F = 3;   // X3F: 3-term forward GEMMs, single-term backward GEMMs
// kind::tf32: activations are fp32 words with TF32-rounded bits, one per TMEM column; an accumulator is
// overwritten in place by the next layer's operand (X = columns 0..127 of the chain, Y = 128..255).
// kind::f16 : activations are fp16 pairs, two per column, so an operand takes half the columns of the
// accumulator it was computed from and cannot be written in place (another thread's accumulator
// columns would be hit): operands always go to X[0:64], accumulators to Y or X[64:128].
// 3-term mode (FMT_F16X3): every operand is the sum of two fp16 numbers, hi = fp16(v) and lo = fp16(v - hi)
// (~21 significant bits); a product is evaluated as hi*hi + lo*hi + hi*lo in the fp32 accumulator -- three
// times the MMAs of FMT_F16, fp32-grade results.  The residual operand sits 64 columns above the main one
// (X[64:128]), so every accumulator -- D3 included -- goes to Y.
// Mixed mode (FMT_F16X3F, the default arithmetic): the forward GEMMs as FMT_F16X3, the backward GEMMs as FMT_F16.
// Single-term backward GEMMs leave X[64:128] idle, which is where the dE/dx operand of the chain's NEXT item is
// stored while B2 of the current item still runs (G_AHEAD in the backward loop): B3 then reads X[64:96].
template <int FMT>
__device__ __forceinline__ OpInfo op_info(int op) {
  if (FMT != FMT_TF32) {
    const int d3 = (FMT == FMT_F16X3 || FMT == FMT_F16X3F) ? 128 : 64;
    switch (op) {
      case 0: return {OFF_W2_H, 2, 128, 4, 0, 128, OFF_W2_HL};     // F2: D2(Y) = A1(X[0:64]) * W2^T
      case 1: return {OFF_W3_H, 1, 64, 8, 0, d3, OFF_W3_HL};       // F3: D3(X[64:128] | Y[0:64]) = A2(X[0:64]) * W3^T
      case 2: return {OFF_W3T_H, 1, 128, 4, (FMT == FMT_F16X3 || !VLG_TC_G_AHEAD) ? 0 : 64, 128, OFF_W3T_HL};   // B3: D4(Y) = G(X[0:32] | X[64:96]) * W3
      default: return {OFF_W2T_H, 2, 128, 4, 0, 128, OFF_W2T_HL};  // B2: D5(Y) = A4(X[0:64]) * W2
    }
  }
  switch (op) {
    case 0: return {OFF_W2_UMMA, 4, 128, 4, 0, 128, 0};    // F2: D2(Y) = A1(X) * W2^T
    case 1: return {OFF_W3_UMMA, 2, 64, 8, 128, 0, 0};     // F3: D3(X[0:64]) = A2(Y) * W3^T
    case 2: return {OFF_W3T_UMMA, 2, 128, 4, 0, 128, 0};   // B3: D4(Y) = G(X[0:64]) * W3
    default: return {OFF_W2T_UMMA, 4, 128, 4, 128, 0, 0};  // B2: D5(X) = A4(Y) * W2
  }
}
// hi / lo fp16 pairs of two fp32 values: hi = fp16(v), lo = fp16(v - hi).  The residual v - hi is exact in fp32 and
// comes from one mixed-precision FMA per element (fma.rn.f32.f16: hi * -1 + v, SASS FHFMA) instead of a convert back
// and a subtract -- 4 instructions per pair instead of 6, same bits.
__device__ __forceinline__ void pack_hilo_h2(float a, float b, uint32_t& hi, uint32_t& lo) {
  float ra, rb;
  asm("{\n\t.reg .b16 l, u, m1;\n\t"
      "cvt.rn.f16x2.f32 %0, %4, %3;\n\t"
      "mov.b32 {l, u}, %0;\n\t"
      "mov.b16 m1, 0xBC00;\n\t"
      "fma.rn.f32.f16 %1, l, m1, %3;\n\t"
      "fma.rn.f32.f16 %2, u, m1, %4;\n\t}"
      : "=&r"(hi), "=f"(ra), "=f"(rb)
      : "f"(a), "f"(b));
  asm("cvt.rn.f16x2.f32 %0, %2, %1;" : "=r"(lo) : "f"(ra), "f"(rb));
}
// two fp32 -> one fp16x2 word (round-to-nearest; lo half = first argument), optionally through relu
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
  const __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t pack_relu_h2(float a, float b) {
  // one instruction: round-to-nearest convert of both values with the ReLU clamp built in
  uint32_t r;
  asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}

// round-to-nearest to TF32 for finite values: the tensor core ignores the 13 low mantissa bits
__device__ __forceinline__ uint32_t tf32_round_bits(uint32_t b) { return b + 0x1000u; }
// relu, then TF32 round-to-nearest on the bit pattern.  (An integer-max formulation,
// max(int(bits + 0x1000), 0), produced wrong results when combined with the packed f32x2
// intrinsics under nvcc 12.9 -- keep the float max.)
__device__ __forceinline__ uint32_t relu_tf32(float v) { return __float_as_uint(fmaxf(v, 0.f)) + 0x1000u; }

}  // namespace
}  // namespace vlg
