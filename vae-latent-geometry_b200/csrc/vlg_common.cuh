// Shared device helpers and the packed-decoder layout.  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "vlg_kernels.h"

namespace vlg {

constexpr int H = 128;          // hidden width of the decoder MLP (src/train.py:80-85)
constexpr int XP = 64;          // padded width of the W3 blocks; X itself is <= 52 (XD_STRIDE / DIFF_STRIDE); tasic-pca50: X = 50
constexpr int TILE_ROWS = 128;  // curve points per tile (= MMA M, = TMEM lanes)
constexpr int TILE_SEGS = 127;  // curve segments per tile: adjacent tiles share one point
constexpr int MAX_NPOLY = 8;
constexpr int MAX_KB = MAX_NPOLY + 1;
constexpr int MAX_M = 4;
constexpr int MAX_K = 255;      // decoder index travels as uint8; 255 = "none"

// ---------------------------------------------------------------------------------------
// Packed decoder image (device memory), produced by vlg_pack_decoders.
//   header (256 B) followed by K per-decoder records of DEC_FLOATS floats.
// Per decoder (float offsets):
//   SMALL   : W1[:,0][128] | W1[:,1][128] | b1[128] | b2[128] | b3[64]    (576 floats)
//   W2T     : [in 128][out 128]    fp32, B operand of the SIMT forward GEMM
//   W2      : [out 128][in 128]    fp32, B operand of the SIMT backward GEMM
//   W3T     : [in 128][out 64]     fp32 (cols >= X are zero)
//   W3      : [out 64][in 128]     fp32 (rows >= X are zero)
//   tcgen05 B-operand images, canonical no-swizzle K-major layout img[k/4][n][k%4]
//   (8x16B core matrices; SBO = 128 B between 8-row groups, LBO = N*16 B between k-chunks),
//   values pre-rounded to TF32 (round-to-nearest):
//   W2_UMMA  : B[n=out][k=in]  = W2[out][in]   N=128 K=128   (h1 * W2^T)
//   W3_UMMA  : B[n=out][k=in]  = W3[out][in]   N=64  K=128   (h2 * W3^T, rows >= X zero)
//   W3T_UMMA : B[n=in][k=out]  = W3[out][in]   N=128 K=64    (dx  * W3)
//   W2T_UMMA : B[n=in][k=out]  = W2[out][in]   N=128 K=128   (dh2 * W2)
//   the same four matrices as fp16 images (round-to-nearest) for kind::f16,
//   img16[k/8][n][k%8] (16-bit elements: a 16-byte core-matrix row holds 8 k; same SBO / LBO):
//   W2_H, W3_H, W3T_H, W2T_H  (offsets below are in floats; an image of N x K halves takes N*K/2)
//   and their fp16 residuals W2_HL, W3_HL, W3T_HL, W2T_HL = fp16(w - fp16(w))
// ---------------------------------------------------------------------------------------
struct PackedHeader {
  uint32_t magic;    // 'VLG1'
  int32_t K, Hdim, X;
  uint32_t dec_floats;
  uint32_t pad[59];
};
static_assert(sizeof(PackedHeader) == 256, "header must be 256 bytes");
constexpr uint32_t PACK_MAGIC = 0x31474c56u;

constexpr int OFF_W1X = 0;    // W1[c][0], c < 128
constexpr int OFF_W1Y = 128;  // W1[c][1]
constexpr int OFF_B1 = 256;
constexpr int OFF_B2 = 384;
constexpr int OFF_B3 = 512;
constexpr int OFF_W2T = 576;
constexpr int OFF_W2 = OFF_W2T + H * H;
constexpr int OFF_W3T = OFF_W2 + H * H;
constexpr int OFF_W3 = OFF_W3T + H * XP;
constexpr int OFF_W2_UMMA = OFF_W3 + XP * H;
constexpr int OFF_W3_UMMA = OFF_W2_UMMA + H * H;
constexpr int OFF_W3T_UMMA = OFF_W3_UMMA + XP * H;
constexpr int OFF_W2T_UMMA = OFF_W3T_UMMA + XP * H;
constexpr int OFF_W2_H = OFF_W2T_UMMA + H * H;
constexpr int OFF_W3_H = OFF_W2_H + H * H / 2;
constexpr int OFF_W3T_H = OFF_W3_H + XP * H / 2;
constexpr int OFF_W2T_H = OFF_W3T_H + XP * H / 2;
// residual images fp16(w - fp16(w)) in the same layout, for the 3-term split mode (fp32-grade on the tensor pipe)
constexpr int OFF_W2_HL = OFF_W2T_H + H * H / 2;
constexpr int OFF_W3_HL = OFF_W2_HL + H * H / 2;
constexpr int OFF_W3T_HL = OFF_W3_HL + XP * H / 2;
constexpr int OFF_W2T_HL = OFF_W3T_HL + XP * H / 2;
constexpr int DEC_FLOATS = OFF_W2T_HL + H * H / 2;
static_assert(DEC_FLOATS % 64 == 0 && OFF_W2_UMMA % 4 == 0, "images must stay 16-byte aligned");

// device-side check of the header against what the caller said it packed (flags VLG_STATUS_BAD_PACKED = 4)
__device__ __forceinline__ bool packed_header_ok(const void* packed, int K_total, int X) {
  const PackedHeader* h = reinterpret_cast<const PackedHeader*>(packed);
  return h->magic == PACK_MAGIC && h->K == K_total && h->X == X && h->Hdim == H && h->dec_floats == uint32_t(DEC_FLOATS);
}

__host__ __device__ inline const float* dec_ptr(const void* packed, int k) {
  return reinterpret_cast<const float*>(reinterpret_cast<const char*>(packed) + sizeof(PackedHeader)) +
         size_t(k) * DEC_FLOATS;
}

// ---------------------------------------------------------------------------------------
// Philox4x32-10: counter-based decoder draws.  Same definition as
// oracle/geodesic_oracle.py:counter_draws (counter = (segment, step, curve id, m/2),
// key = seed; word w -> decoder index (w*K)>>32).
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
    uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += W0;
    k.y += W1;
  }
  return c;
}

// Decoder index for (curve, step, MC sample m, role, segment).
__device__ __forceinline__ void counter_draws4(uint64_t seed, uint32_t curve, uint32_t step,
                                               uint32_t seg, uint32_t mpair, uint32_t K,
                                               uint32_t out[4]) {
  uint4 w = philox4x32_10(make_uint4(seg, step, curve, mpair),
                          make_uint2(uint32_t(seed), uint32_t(seed >> 32)));
  out[0] = __umulhi(w.x, K);
  out[1] = __umulhi(w.y, K);
  out[2] = __umulhi(w.z, K);
  out[3] = __umulhi(w.w, K);
}

// ---------------------------------------------------------------------------------------
// Spline helpers (src/optimize.py:22-35).
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void seg_coords(float t, int n_poly, int& seg, float& u) {
  float tn = t * float(n_poly);
  int s = int(floorf(tn));
  seg = s < n_poly - 1 ? s : n_poly - 1;
  u = tn - float(seg);
}

// z = (1-t) a + t b + sum_i u^i coef[seg][i]   (coef = basis @ omega, [n_poly][4][2])
__device__ __forceinline__ float2 spline_point(float t, int n_poly, const float* coef, float2 a,
                                               float2 b) {
  int seg;
  float u;
  seg_coords(t, n_poly, seg, u);
  const float* c = coef + seg * 8;
  float u2 = u * u, u3 = u2 * u;
  float px = c[0] + u * c[2] + u2 * c[4] + u3 * c[6];
  float py = c[1] + u * c[3] + u2 * c[5] + u3 * c[7];
  float omt = 1.0f - t;
  return make_float2(omt * a.x + t * b.x + px, omt * a.y + t * b.y + py);
}

// Row of the design matrix P[t][k] = sum_i u^i basis[4 seg + i][k].
__device__ __forceinline__ void design_row(float t, int n_poly, int Kb, const float* basis, float* P) {
  int seg;
  float u;
  seg_coords(t, n_poly, seg, u);
  float u2 = u * u, u3 = u2 * u;
  const float* r = basis + seg * 4 * Kb;
#pragma unroll
  for (int k = 0; k < MAX_KB; ++k)
    if (k < Kb) P[k] = r[k] + u * r[Kb + k] + u2 * r[2 * Kb + k] + u3 * r[3 * Kb + k];
}

// Adam scalars for 1-based step s, as torch computes them in double (torch/optim/adam.py):
// step_size = lr / (1 - beta1^s), denom = sqrt(v) / sqrt(1 - beta2^s) + eps.
struct AdamScalars {
  float step_size, bc2_sqrt;
};
__device__ inline AdamScalars adam_scalars(int step, double lr, double beta1, double beta2) {
  double bc1 = 1.0 - pow(beta1, double(step));
  double bc2 = 1.0 - pow(beta2, double(step));
  AdamScalars s;
  s.step_size = float(lr / bc1);
  s.bc2_sqrt = float(sqrt(bc2));
  return s;
}

// one_minus_b1 = float(1 - beta1), beta2f = float(beta2), one_minus_b2 = float(1 - beta2):
// rounded from the double expressions exactly as torch hands them to lerp_/mul_/addcmul_.
__device__ __forceinline__ void adam_update(float& p, float& m, float& v, float g, AdamScalars s,
                                            float one_minus_b1, float beta2f, float one_minus_b2,
                                            float eps) {
  m = m + (g - m) * one_minus_b1;
  v = v * beta2f + (one_minus_b2 * g) * g;
  float denom = sqrtf(v) / s.bc2_sqrt + eps;
  p = p - s.step_size * (m / denom);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---------------------------------------------------------------------------------------
// Per-curve step code of both step kernels (vlg_simt.cu, vlg_tc.cu).  `status` is the launch's status word
// (VLG_STATUS_* flags, word [1] of the workspace header).  A curve's optimiser state `om` holds omega, m and v
// at offsets 0, 2 MAX_KB and 4 MAX_KB.
// ---------------------------------------------------------------------------------------
// fp16 operands overflow above 65504: inf/NaN reach the energy (forward), the gradient or omega (backward)
__device__ __forceinline__ void flag_nonfinite(float x, unsigned int* status) {
  if (!(fabsf(x) <= 3.0e38f)) atomicOr(status, unsigned(VLG_STATUS_NONFINITE));
}

// First decoder of curve n's weight set inside `packed`.  Out of range: 0 (memory safety), reported by the
// thread that passes `report`.
__device__ __forceinline__ int curve_dec_base(const StepParams& p, int n, bool report, unsigned int* status) {
  int base = p.dec_base ? p.dec_base[n] : 0;
  if (base < 0 || base + p.K > p.K_total) {
    base = 0;
    if (report) atomicOr(status, unsigned(VLG_STATUS_BAD_PACKED));
  }
  return base;
}

// Explicit draw [n][step][m][role][seg] of draws [N][steps][M][2][T-1].  A value >= K is clamped to K - 1 (memory
// safety) and sets `bad`, which the kernel reports through the status word.  The sizes come as arguments rather than
// through StepParams: the callers store draws as bytes, which may alias a StepParams reference and would force a
// reload of every field per draw, where the kernels keep the sizes in registers.
__device__ __forceinline__ uint8_t explicit_draw(const uint8_t* draws, int steps, int M, int T, int K, int n, int step,
                                                 int m, int role, int seg, bool& bad) {
  uint8_t v = draws[(((size_t(n) * steps + step) * M + m) * 2 + role) * size_t(T - 1) + seg];
  if (v >= K) { v = uint8_t(K - 1); bad = true; }
  return v;
}

// Energy of curve n at `step` from its sums over the M samples: the trace entry and, at the launch's last step,
// the energy and poly-line length outputs.
__device__ __forceinline__ void write_energy(const StepParams& p, int n, int step, float e_sum, float l_sum,
                                             unsigned int* status) {
  const float E = e_sum / float(p.M);
  flag_nonfinite(E, status);
  if (p.energy_trace) p.energy_trace[size_t(step) * p.N + n] = E;
  if (step == p.steps - 1) {
    if (p.energy_last) p.energy_last[n] = E;
    if (p.length_out) p.length_out[n] = l_sum / float(p.M);
  }
}

// Component c of curve n's gradient output (EnergyGrad): dE/d(omega) for c < 2 Kb, then dE/da, dE/db.
__device__ __forceinline__ void write_grad(const StepParams& p, int n, int c, float g, unsigned int* status) {
  const int Kb = p.Kb;
  flag_nonfinite(g, status);
  if (c < 2 * Kb) p.grad_omega[size_t(n) * 2 * Kb + c] = g;
  else if (c < 2 * Kb + 2) p.grad_a[2 * n + c - 2 * Kb] = g;
  else p.grad_b[2 * n + c - 2 * Kb - 2] = g;
}

// One optimiser step of coefficient c = 2 k + d of a curve (end points a, b; coef = basis @ omega): the energy
// gradient g_energy plus that of the end-point penalty w |z(t_end) - b|^2, then Adam on om.
__device__ __forceinline__ void penalty_adam_step(const StepParams& p, int step, int c, float g_energy,
                                                  const float* basis, const float* coef, float2 pa, float2 pb,
                                                  float* om) {
  const int k = c >> 1, d = c & 1;
  const float tend = p.t[p.T - 1];
  float P[MAX_KB];
  design_row(tend, p.n_poly, p.Kb, basis, P);
  const float2 ze = spline_point(tend, p.n_poly, coef, pa, pb);
  const float err = d == 0 ? ze.x - pb.x : ze.y - pb.y;
  const float g = g_energy + (2.0f * p.penalty_w) * err * P[k];
  AdamScalars sc = adam_scalars(p.step0 + step + 1, p.lr, p.beta1, p.beta2);
  float w = om[c], mm = om[2 * MAX_KB + c], vv = om[4 * MAX_KB + c];
  adam_update(w, mm, vv, g, sc, p.one_minus_b1, p.beta2f, p.one_minus_b2, p.eps);
  om[c] = w;
  om[2 * MAX_KB + c] = mm;
  om[4 * MAX_KB + c] = vv;
}

// omega, m and v of coefficient c of curve n back to memory (Optimize)
__device__ __forceinline__ void write_back(const StepParams& p, int n, int c, const float* om, unsigned int* status) {
  const size_t o = size_t(n) * 2 * p.Kb + c;
  p.omega[o] = om[c];
  p.adam_m[o] = om[2 * MAX_KB + c];
  p.adam_v[o] = om[4 * MAX_KB + c];
  flag_nonfinite(om[c], status);
}

}  // namespace vlg
