// Decoder ensemble as a differentiable op (vlg_decode / vlg_decode_backward):
//   x[k, p, :] = f_k(z[p])                                     k = 0 .. K_active-1, f_k = 2 -> 128 -> ReLU -> 128 -> ReLU -> X
//   dz[p]      = sum_k W1^T (m1 . W2^T (m2 . W3^T dx[k, p]))   over k in increasing order
// (`torch.stack([d(z).mean for d in decoders])`, src/optimize.py:50, and its input gradient).
//
// Tensor-core kernel (tc_decode_kernel<FMT, MODE>).  Persistent CTAs, two per SM, walk 128-point tiles; for every tile
// the decoders run one after the other as "items" of one chain of 256 TMEM columns (rows = the 128 TMEM lanes).  The
// GEMMs, their operand formats and TMEM columns are those of the step kernel (vlg_tc_ops.cuh: op_info); the B operands
// are the packed weight images, streamed into a shared-memory ring by 1-D bulk copies.
//   forward item : layer 1 (CUDA cores, fp32) -> F2 -> relu(+b2) -> F3 -> +b3 -> x
//   backward item: layer 1 (masks m1) -> F2 (masks m2 only) -> B3 with the dx row -> mask m2 -> B2 -> mask m1 ->
//                  contraction with W1^T (CUDA cores, fp32) -> dz
// The backward recomputes the masks, so nothing is kept between the two calls.  Warp 0 issues the bulk copies, warp 1
// the MMAs (one elected lane), warps 2-5 are the epilogue with one thread per row: a thread owns its row's TMEM lane in
// every phase, and each point's dz is a register sum over the decoders in order (no atomics, no timing dependence).
// The second CTA of an SM is the second chain: its items overlap the first CTA's epilogue phases.
//
// dx scale.  The caller chooses the scale of dx (a loss divided by N, a loss scale, ...), so each row of dx is
// normalised by a power of two 2^(6 - e), e = ilogb(max_c |dx[k, p, c]|), before it is rounded to an operand, and dz
// is multiplied by 2^(e - 6) in fp32.  Every GEMM acts row by row and the masks do not depend on dx, so the scaling is
// exact: decode_backward(2^s dx) has exactly the bits of 2^s decode_backward(dx).  An all-zero row contributes 0.
//
// fp32 CUDA-core kernels (simt_decode_kernel<MODE>) for precision fp32 and K_active > 128: the structure of
// std_norm_kernel (vlg_pack.cu), 32 points per 128-thread block, thread j = hidden unit j.
//
// Expected ensemble energy (vlg_expected_energy) of curves z [T][N][2], point p = t * N + n, on the same kernels:
//   Mean       every decoder's forward; mu[p] = (1/K) sum_k x[k, p], summed in decoder order in the mean row itself
//   Energy     every decoder's forward again: e[p] = c_t V_t + ||mu_{t+1} - mu_t||^2 (no second term at t = T-1),
//              V_t = (1/K) sum_k ||x[k, p] - mu_t||^2 around the mean of the first pass
//   EnergyGrad Energy, and per item B3 B2 on the dE/dx row (x - mu_{t-1}) + (x - mu_{t+1}) (one term at the ends):
//              dz[p] = (2/K) sum_k J_k^T (c_t x[k, p] - mu_{t-1} - mu_{t+1})
// then curve_sum_kernel: energy[n] = sum_t e[t * N + n] in increasing t.
#include <cuda_fp16.h>

#include "../../include/vlg.h"
#include "vlg_common.cuh"
#include "vlg_kernels.h"
#include "vlg_tc_ops.cuh"
#include "vlg_tcgen05.cuh"

namespace vlg {

namespace {

using namespace tc;

constexpr int DEC_THREADS = 192;     // producer warp, MMA warp, 4 epilogue warps
constexpr int DEC_STAGES = 6;        // 16 KB weight stages in the ring
constexpr int DEC_TMEM_COLS = 256;   // one chain: X = columns 0..127, Y = 128..255
constexpr int DEC_BAR_BYTES = 256;
constexpr size_t DEC_SMEM = size_t(DEC_STAGES) * STAGE_BYTES + DEC_BAR_BYTES;
constexpr int DEC_CTAS_PER_SM = 2;

// What a launch computes (the kernels' template parameter):
//   Forward    x[k, p, :] = f_k(z[p])                                    (vlg_decode)
//   Backward   dz[p] = sum_k J_k(z[p])^T dx[k, p]                         (vlg_decode_backward)
//   Mean       mu[p] = (1/K) sum_k f_k(z[p])                             (vlg_expected_energy, first pass)
//   Energy     e[p] = c_t V_t + ||mu_{t+1} - mu_t||^2 around that mean  (second pass)
//   EnergyGrad e[p] and dz[p] = dE/dz_t = (2/K) sum_k J_k^T (c_t x_k - mu_{t-1} - mu_{t+1})
enum class DecodeMode { Forward, Backward, Mean, Energy, EnergyGrad };

struct DecodeArgs {
  const void* packed;
  int K_total, X, K, P;
  const float* z;       // [P][2]
  const float* dx;      // [K][P][X] (backward)
  float* x;             // [K][P][X] (forward)
  float* dz;            // [P][2]    (backward, EnergyGrad)
  unsigned int* status; // word [1] of the workspace
  // expected energy: the points are curves z [T][N][2], p = t * N + n (fields after the decode ones: those keep their
  // parameter offsets, so the decode kernels compile as before)
  int N;
  float* mu;            // [P][X] ensemble mean: written by Mean, read by Energy / EnergyGrad
  float* e;             // [P]    per-point energy terms
};

__device__ __forceinline__ bool finite32(float v) { return fabsf(v) <= 3.0e38f; }
// dE/dx of one output of decoder k at a curve point, up to the factor 2 / K, as a sum of fp32 differences:
// (x - mu_{t-1}) + (x - mu_{t+1}) inside the curve (inner), the one existing term x - mu1 at its ends
__device__ __forceinline__ float expected_dedx(float x, const float* mu1, const float* mu2, bool inner, int c) {
  return inner ? (x - __ldg(mu1 + c)) + (x - __ldg(mu2 + c)) : x - __ldg(mu1 + c);
}

// the GEMMs of item op j: backward F2 B3 B2, every other mode F2 F3 (EnergyGrad: F2 F3 B3 B2) (op_info numbering)
template <bool BWD>
__device__ __forceinline__ int item_op(int j) { return BWD ? (j == 0 ? 0 : j + 1) : j; }

// G columns c0 .. c0 + 7 (normalised dE/dx values of one row) -> B3's A operand
template <int FMT>
__device__ __forceinline__ void store_g8(uint32_t colX, int c0, const float (&g)[8]) {
  constexpr bool X3B = FMT == FMT_F16X3;
  const OpInfo ob3 = op_info<FMT>(2);
  if (FMT != FMT_TF32) {
    uint32_t v[4], vl[X3B ? 4 : 1];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (X3B) pack_hilo_h2(g[2 * j], g[2 * j + 1], v[j], vl[j]);
      else v[j] = pack_h2(g[2 * j], g[2 * j + 1]);
    }
    tmem_st4(colX + ob3.a_col + c0 / 2, v);
    if (X3B) tmem_st4(colX + ob3.a_col + 64 + c0 / 2, reinterpret_cast<uint32_t(&)[4]>(vl));
  } else {
    uint32_t v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = tf32_round_bits(__float_as_uint(g[j]));
    tmem_st8(colX + ob3.a_col + c0, v);
  }
}

template <int FMT, DecodeMode MODE>
__global__ void __launch_bounds__(DEC_THREADS, DEC_CTAS_PER_SM) tc_decode_kernel(DecodeArgs a) {
  constexpr bool F16 = FMT != FMT_TF32;
  constexpr bool X3F = FMT == FMT_F16X3 || FMT == FMT_F16X3F;   // 3-term F2, F3
  constexpr bool X3B = FMT == FMT_F16X3;                        // 3-term B3, B2
  constexpr bool BWD = MODE == DecodeMode::Backward;
  constexpr bool EGRAD = MODE == DecodeMode::EnergyGrad;
  constexpr bool EXPECT = MODE == DecodeMode::Energy || EGRAD;  // V_t and e_t around the mean of a Mean launch
  constexpr int NOPS = BWD ? 3 : EGRAD ? 4 : 2;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned char* ring = smem_raw;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + DEC_STAGES * STAGE_BYTES);
  uint64_t* empty = full + DEC_STAGES;
  uint64_t* a_ready = empty + DEC_STAGES;   // the epilogue has stored the next GEMM's A operand (one arrival per warp)
  uint64_t* acc_ready = a_ready + 1;        // the GEMM's accumulator is complete
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_ready + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ntiles = (a.P + 127) / 128;
  const int K = a.K;

  if (tid == 0) {
    for (int i = 0; i < DEC_STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(a_ready, 4);
    mbar_init(acc_ready, 1);
    fence_mbar_init();
  }
  if (blockIdx.x == 0 && tid == 32 && !packed_header_ok(a.packed, a.K_total, a.X))
    atomicOr(a.status, unsigned(VLG_STATUS_BAD_PACKED));
  if (warp == 1) tmem_alloc(tmem_slot, DEC_TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    // ================= weight producer: the B images of every GEMM, in issue order =================
    if (lane == 0) {
      int slot = 0;
      uint32_t ph = 0;
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
        for (int k = 0; k < K; ++k)
          for (int j = 0; j < NOPS; ++j) {
            const int op = item_op<BWD>(j);
            const OpInfo oi = op_info<FMT>(op);
            const bool x3 = op < 2 ? X3F : X3B;
            const char* src = reinterpret_cast<const char*>(dec_ptr(a.packed, k) + oi.img_off);
            const char* src_lo = reinterpret_cast<const char*>(dec_ptr(a.packed, k) + oi.img_lo);
            // 3-term: the stages of the main image, then those of the residual image
            for (int st = 0; st < (x3 ? 2 : 1) * oi.nstages; ++st) {
              const char* from = st < oi.nstages ? src + size_t(st) * STAGE_BYTES : src_lo + size_t(st - oi.nstages) * STAGE_BYTES;
              mbar_wait(&empty[slot], ph ^ 1);
              mbar_expect_tx(&full[slot], STAGE_BYTES);
              bulk_g2s(ring + slot * STAGE_BYTES, from, STAGE_BYTES, &full[slot]);
              if (++slot == DEC_STAGES) { slot = 0; ph ^= 1; }
            }
          }
    }
  } else if (warp == 1) {
    // ================= MMA issuer (whole warp, one elected lane takes effect) =================
    const uint32_t leader = elect_one();
    int slot = 0;
    uint32_t ph = 0, ph_a = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
      for (int k = 0; k < K; ++k)
        for (int j = 0; j < NOPS; ++j) {
          const int op = item_op<BWD>(j);
          const OpInfo oi = op_info<FMT>(op);
          const bool x3 = op < 2 ? X3F : X3B;
          const uint32_t idesc = F16 ? umma_idesc_f16(oi.n) : umma_idesc_tf32(oi.n, 0);
          mbar_wait(a_ready, ph_a);
          ph_a ^= 1;
          tc_fence_after();
          for (int st = 0; st < (x3 ? 2 : 1) * oi.nstages; ++st) {
            mbar_wait(&full[slot], ph);
            tc_fence_after();
            const uint32_t sbase = smem_u32(ring + slot * STAGE_BYTES);
            const bool w_lo = x3 && st >= oi.nstages;   // this stage holds residual weights
            const int kst = w_lo ? st - oi.nstages : st;
            // main weights: main operand (and, 3-term, the residual operand 64 columns up); residual weights: main operand
            for (int term = 0; term < ((x3 && !w_lo) ? 2 : 1); ++term)
              for (int ks = 0; ks < oi.nk; ++ks) {
                const uint64_t desc = umma_smem_desc(sbase + uint32_t(ks) * 2u * uint32_t(oi.n) * 16u, uint32_t(oi.n) * 16u, 128u);
                const uint32_t a_addr = tmem + oi.a_col + uint32_t(term * 64) + uint32_t((kst * oi.nk + ks) * 8);
                const uint32_t accum = (st | ks | term) ? 1u : 0u;
                if (F16)
                  umma_f16_ts_elect(tmem + oi.d_col, a_addr, desc, idesc, accum, leader);
                else
                  umma_tf32_ts_elect(tmem + oi.d_col, a_addr, desc, idesc, accum, leader);
              }
            umma_commit_elect(&empty[slot], leader);
            if (++slot == DEC_STAGES) { slot = 0; ph ^= 1; }
          }
          umma_commit_elect(acc_ready, leader);
        }
  } else {
    // ================= epilogue: one thread per row (TMEM lane) =================
    const int row = (warp & 3) * 32 + lane;
    const uint32_t colX = tmem + (uint32_t((warp & 3) * 32) << 16), colY = colX + 128u;
    const int X = a.X;
    const size_t P = size_t(a.P);
    uint32_t ph_acc = 0;
    bool bad = false;
    auto operand_ready = [&]() {
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(a_ready);
    };
    auto acc_wait = [&]() {
      mbar_wait(acc_ready, ph_acc);
      ph_acc ^= 1;
      tc_fence_after();
    };
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      const int p = tile * 128 + row;
      const bool valid = p < a.P;
      const float2 z = valid ? reinterpret_cast<const float2*>(a.z)[p] : make_float2(0.f, 0.f);
      // (the ReLUs map NaN to 0, so a non-finite point need not reach x or dz: it is flagged itself)
      bad |= !finite32(z.x) || !finite32(z.y);
      const float2 zx2 = make_float2(z.x, z.x), zy2 = make_float2(z.y, z.y);
      float dzx = 0.f, dzy = 0.f;
      // expected energy: point p = t * N + n of its curve, the mean rows of p and of its neighbours t - 1, t + 1
      const int t = EXPECT && valid ? p / a.N : 0;
      const bool has_prev = t > 0, has_next = EXPECT && t < a.P / a.N - 1;   // T >= 2: at least one of them
      const size_t nbr = size_t(a.N) * size_t(X);
      const float* mu0 = a.mu + size_t(valid ? p : 0) * size_t(X);
      const float* mu1 = has_prev ? mu0 - nbr : mu0 + nbr;       // one neighbour; inside the curve mu0 + nbr is the other
      const bool inner = has_prev && has_next;
      float vsum = 0.f;   // sum_k ||x_k - mu_t||^2
      for (int k = 0; k < K; ++k) {
        const float* d = dec_ptr(a.packed, k);
        // ---- layer 1 (CUDA cores, fp32) -> A1: X[0:64] fp16 pairs (+ residuals X[64:128]) | X[0:128] tf32 ----
        uint32_t m1[4];
#pragma unroll
        for (int hh = 0; hh < 4; ++hh) {   // 32 hidden units per pass
          uint32_t v[32], vl[X3F ? 16 : 1];
          uint32_t mb = 0;
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const int c = 32 * hh + j;
            const float4 wx = __ldg(reinterpret_cast<const float4*>(d + OFF_W1X + c));
            const float4 wy = __ldg(reinterpret_cast<const float4*>(d + OFF_W1Y + c));
            const float4 bb = __ldg(reinterpret_cast<const float4*>(d + OFF_B1 + c));
            const float2 h0 = __ffma2_rn(make_float2(wy.x, wy.y), zy2, __ffma2_rn(make_float2(wx.x, wx.y), zx2, make_float2(bb.x, bb.y)));
            const float2 h1 = __ffma2_rn(make_float2(wy.z, wy.w), zy2, __ffma2_rn(make_float2(wx.z, wx.w), zx2, make_float2(bb.z, bb.w)));
            if (BWD || EGRAD) mb |= (h0.x > 0.f ? 1u : 0u) << j | (h0.y > 0.f ? 2u : 0u) << j | (h1.x > 0.f ? 4u : 0u) << j | (h1.y > 0.f ? 8u : 0u) << j;
            if (X3F) {
              pack_hilo_h2(fmaxf(h0.x, 0.f), fmaxf(h0.y, 0.f), v[j >> 1], vl[j >> 1]);
              pack_hilo_h2(fmaxf(h1.x, 0.f), fmaxf(h1.y, 0.f), v[(j >> 1) + 1], vl[(j >> 1) + 1]);
            } else if (F16) {
              v[j >> 1] = pack_relu_h2(h0.x, h0.y);
              v[(j >> 1) + 1] = pack_relu_h2(h1.x, h1.y);
            } else {
              v[j] = relu_tf32(h0.x); v[j + 1] = relu_tf32(h0.y); v[j + 2] = relu_tf32(h1.x); v[j + 3] = relu_tf32(h1.y);
            }
          }
          m1[hh] = mb;
          if (F16) {
            tmem_st16(colX + 16 * hh, reinterpret_cast<uint32_t(&)[16]>(v));
            if (X3F) tmem_st16(colX + 64 + 16 * hh, reinterpret_cast<uint32_t(&)[16]>(vl));
          } else {
            tmem_st32(colX + 32 * hh, v);
          }
        }
        operand_ready();
        // ---- F2 done: D2 (Y) + b2 -> forward: A2 (X[0:64] (+ X[64:128]) | Y in place); backward: masks m2 ----
        acc_wait();
        uint32_t m2[4];
#pragma unroll
        for (int hh = 0; hh < 4; ++hh) {
          uint32_t v[32], vl[X3F ? 16 : 1];
          tmem_ld32_sync(colY + 32 * hh, v);
          uint32_t mb = 0;
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const float4 b0 = __ldg(reinterpret_cast<const float4*>(d + OFF_B2 + 32 * hh + j));
            const float2 p0 = __fadd2_rn(make_float2(__uint_as_float(v[j]), __uint_as_float(v[j + 1])), make_float2(b0.x, b0.y));
            const float2 p1 = __fadd2_rn(make_float2(__uint_as_float(v[j + 2]), __uint_as_float(v[j + 3])), make_float2(b0.z, b0.w));
            if constexpr (EGRAD)
              mb |= (p0.x > 0.f ? 1u : 0u) << j | (p0.y > 0.f ? 2u : 0u) << j | (p1.x > 0.f ? 4u : 0u) << j | (p1.y > 0.f ? 8u : 0u) << j;
            if (BWD) {
              mb |= (p0.x > 0.f ? 1u : 0u) << j | (p0.y > 0.f ? 2u : 0u) << j | (p1.x > 0.f ? 4u : 0u) << j | (p1.y > 0.f ? 8u : 0u) << j;
            } else if (X3F) {   // pairs go to v[0:16]: slots j/2, j/2+1 <= j were consumed already
              uint32_t a0, a1;
              pack_hilo_h2(fmaxf(p0.x, 0.f), fmaxf(p0.y, 0.f), a0, vl[j >> 1]);
              pack_hilo_h2(fmaxf(p1.x, 0.f), fmaxf(p1.y, 0.f), a1, vl[(j >> 1) + 1]);
              v[j >> 1] = a0;
              v[(j >> 1) + 1] = a1;
            } else if (F16) {
              const uint32_t a0 = pack_relu_h2(p0.x, p0.y), a1 = pack_relu_h2(p1.x, p1.y);
              v[j >> 1] = a0;
              v[(j >> 1) + 1] = a1;
            } else {
              v[j] = relu_tf32(p0.x); v[j + 1] = relu_tf32(p0.y); v[j + 2] = relu_tf32(p1.x); v[j + 3] = relu_tf32(p1.y);
            }
          }
          m2[hh] = mb;
          if (!BWD) {
            if (F16) {
              tmem_st16(colX + 16 * hh, reinterpret_cast<uint32_t(&)[16]>(v));
              if (X3F) tmem_st16(colX + 64 + 16 * hh, reinterpret_cast<uint32_t(&)[16]>(vl));
            } else {
              tmem_st32(colY + 32 * hh, v);
            }
          }
        }
        float amax_g = 0.f;   // EnergyGrad: the largest |dE/dx| of the row
        if (!BWD) {
          operand_ready();
          // ---- F3 done: D3 + b3 -> x[k, p, :] ----
          acc_wait();
          const uint32_t d3 = X3F ? colY : colX + (F16 ? 64u : 0u);
          if constexpr (MODE == DecodeMode::Forward) {
            float* xo = a.x + (size_t(k) * P + size_t(valid ? p : 0)) * size_t(X);
#pragma unroll
            for (int c0 = 0; c0 < 64; c0 += 32) {
              uint32_t v[32];
              tmem_ld32_sync(d3 + c0, v);
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                const float4 bb = __ldg(reinterpret_cast<const float4*>(d + OFF_B3 + c0 + j));
                const float o[4] = {__uint_as_float(v[j]) + bb.x, __uint_as_float(v[j + 1]) + bb.y,
                                    __uint_as_float(v[j + 2]) + bb.z, __uint_as_float(v[j + 3]) + bb.w};
#pragma unroll
                for (int e = 0; e < 4; ++e)
                  if (valid && c0 + j + e < X) {
                    xo[c0 + j + e] = o[e];
                    bad |= !finite32(o[e]);
                  }
              }
            }
          } else if constexpr (MODE == DecodeMode::Mean) {
            // mu row += x (the row is this thread's alone), divided by K after the last decoder
            float* mr = a.mu + size_t(valid ? p : 0) * size_t(X);
#pragma unroll
            for (int c0 = 0; c0 < 64; c0 += 32) {
              uint32_t v[32];
              tmem_ld32_sync(d3 + c0, v);
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (valid && c0 + j < X) {
                  const float x = __uint_as_float(v[j]) + __ldg(d + OFF_B3 + c0 + j);
                  const float s = k == 0 ? x : mr[c0 + j] + x;
                  mr[c0 + j] = k == K - 1 ? s / float(K) : s;
                  if (k == K - 1) bad |= !finite32(s);
                }
            }
          } else {
            // ||x - mu_t||^2; EnergyGrad: the largest |dE/dx| of the row.  8 columns at a time, not unrolled: the
            // mean rows' loads of a wider chunk would not fit the registers
#pragma unroll 1
            for (int c0 = 0; c0 < X; c0 += 8) {
              uint32_t v[8];
              tmem_ld8_sync(d3 + c0, v);
#pragma unroll
              for (int j = 0; j < 8; ++j)
                if (valid && c0 + j < X) {
                  const float x = __uint_as_float(v[j]) + __ldg(d + OFF_B3 + c0 + j);
                  const float dm = x - __ldg(mu0 + c0 + j);
                  vsum = fmaf(dm, dm, vsum);
                  if (EGRAD) amax_g = fmaxf(amax_g, fabsf(expected_dedx(x, mu1, mu0 + nbr, inner, c0 + j)));
                }
            }
          }
          if constexpr (!EGRAD) continue;
        }
        // ---- G = the dx row of (k, p), normalised by 2^(6 - e) -> B3's A operand ----
        const float* dxr = a.dx + (size_t(k) * P + size_t(valid ? p : 0)) * size_t(X);
        float amax = 0.f;
        if constexpr (EGRAD)
          amax = amax_g;
        else if (valid)
          for (int c = 0; c < X; ++c) amax = fmaxf(amax, fabsf(__ldg(dxr + c)));
        // (e clamped to [-120, 127]: both scale factors stay normal fp32 numbers)
        const int e = (amax > 0.f && finite32(amax)) ? max(ilogbf(amax), -120) : 6;
        const float sc = ldexpf(1.f, 6 - e), unsc = ldexpf(1.f, e - 6);
        if constexpr (EGRAD) {
          // the row again from D3, chunk by chunk after its columns are read (f16, tf32: G overwrites them)
#pragma unroll 1
          for (int c0 = 0; c0 < 64; c0 += 8) {
            uint32_t v[8];
            tmem_ld8_sync((X3F ? colY : colX + (F16 ? 64u : 0u)) + c0, v);
            float g[8];
#pragma unroll
            for (int j = 0; j < 8; ++j)
              g[j] = (valid && c0 + j < X)
                         ? expected_dedx(__uint_as_float(v[j]) + __ldg(d + OFF_B3 + c0 + j), mu1, mu0 + nbr, inner, c0 + j) * sc
                         : 0.f;
            store_g8<FMT>(colX, c0, g);
          }
        } else {
          const OpInfo ob3 = op_info<FMT>(2);
#pragma unroll
          for (int c0 = 0; c0 < 64; c0 += 32) {
            float g[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) g[j] = (valid && c0 + j < X) ? __ldg(dxr + c0 + j) * sc : 0.f;
            if (F16) {
              uint32_t v[16], vl[X3B ? 16 : 1];
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                if (X3B) pack_hilo_h2(g[2 * j], g[2 * j + 1], v[j], vl[j]);
                else v[j] = pack_h2(g[2 * j], g[2 * j + 1]);
              }
              tmem_st16(colX + ob3.a_col + c0 / 2, v);
              if (X3B) tmem_st16(colX + ob3.a_col + 64 + c0 / 2, reinterpret_cast<uint32_t(&)[16]>(vl));
            } else {
              uint32_t v[32];
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = tf32_round_bits(__float_as_uint(g[j]));
              tmem_st32(colX + ob3.a_col + c0, v);
            }
          }
        }
        operand_ready();
        // ---- B3 done: D4 (Y) masked by m2 -> A4 (X[0:64] (+ X[64:128]) | Y in place) ----
        acc_wait();
#pragma unroll
        for (int hh = 0; hh < 4; ++hh) {
          uint32_t v[32];
          tmem_ld32_sync(colY + 32 * hh, v);
          const uint32_t mb = m2[hh];
          if (F16) {
            uint32_t vl[X3B ? 16 : 1];
#pragma unroll
            for (int j = 0; j < 32; j += 2) {
              const float a0 = ((mb >> j) & 1u) ? __uint_as_float(v[j]) : 0.f;
              const float a1 = ((mb >> (j + 1)) & 1u) ? __uint_as_float(v[j + 1]) : 0.f;
              if (X3B) pack_hilo_h2(a0, a1, v[j >> 1], vl[j >> 1]);
              else v[j >> 1] = pack_h2(a0, a1);   // j/2 <= j: slot already consumed
            }
            tmem_st16(colX + 16 * hh, reinterpret_cast<uint32_t(&)[16]>(v));
            if (X3B) tmem_st16(colX + 64 + 16 * hh, reinterpret_cast<uint32_t(&)[16]>(vl));
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = ((mb >> j) & 1u) ? tf32_round_bits(v[j]) : 0u;
            tmem_st32(colY + 32 * hh, v);
          }
        }
        operand_ready();
        // ---- B2 done: D5 (Y | X) masked by m1, contracted with W1^T in fp32 -> dz of this decoder ----
        acc_wait();
        {
          float2 ax = make_float2(0.f, 0.f), ay = make_float2(0.f, 0.f);
#pragma unroll
          for (int hh = 0; hh < 4; ++hh) {
            uint32_t v[32];
            tmem_ld32_sync((F16 ? colY : colX) + 32 * hh, v);
            const uint32_t mb = m1[hh];
#pragma unroll
            for (int j = 0; j < 32; j += 2) {
              const float2 wx = __ldg(reinterpret_cast<const float2*>(d + OFF_W1X + 32 * hh + j));
              const float2 wy = __ldg(reinterpret_cast<const float2*>(d + OFF_W1Y + 32 * hh + j));
              const float2 dh = make_float2(((mb >> j) & 1u) ? __uint_as_float(v[j]) : 0.f,
                                            ((mb >> (j + 1)) & 1u) ? __uint_as_float(v[j + 1]) : 0.f);
              ax = __ffma2_rn(dh, wx, ax);
              ay = __ffma2_rn(dh, wy, ay);
            }
          }
          dzx += (ax.x + ax.y) * unsc;
          dzy += (ay.x + ay.y) * unsc;
        }
      }
      if (BWD && valid) {
        reinterpret_cast<float2*>(a.dz)[p] = make_float2(dzx, dzy);
        bad |= !finite32(dzx) || !finite32(dzy);
      }
      if (EXPECT && valid) {
        // e_t = c_t V_t + ||mu_{t+1} - mu_t||^2 (the segment that starts at t), c_t = the segments that touch t
        float et = float(int(has_prev) + int(has_next)) * (vsum / float(K));
        if (has_next) {
          float s = 0.f;
          for (int c = 0; c < X; ++c) {
            const float dm = __ldg(mu0 + nbr + c) - __ldg(mu0 + c);
            s = fmaf(dm, dm, s);
          }
          et += s;
        }
        a.e[p] = et;
        bad |= !finite32(et);
      }
      if (EGRAD && valid) {
        const float gx = 2.f * dzx / float(K), gy = 2.f * dzy / float(K);
        reinterpret_cast<float2*>(a.dz)[p] = make_float2(gx, gy);
        bad |= !finite32(gx) || !finite32(gy);
      }
    }
    if (bad) atomicOr(a.status, unsigned(VLG_STATUS_NONFINITE));
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, DEC_TMEM_COLS);
  }
}

// ---- fp32 CUDA-core kernels: 32 points per block, thread j = hidden unit j (and output j < X) ----
constexpr int DSP = 32;

template <DecodeMode MODE>
__global__ void __launch_bounds__(128) simt_decode_kernel(DecodeArgs a) {
  constexpr bool BWD = MODE == DecodeMode::Backward;
  constexpr bool EGRAD = MODE == DecodeMode::EnergyGrad;
  constexpr bool EXPECT = MODE == DecodeMode::Energy || EGRAD;
  __shared__ float h1[DSP][H + 1];   // layer-1 activations; backward: then dh2
  __shared__ float h2[DSP][H + 1];   // forward: layer-2 activations; backward: dx rows [DSP][XP]
  __shared__ float zz[DSP][2];
  __shared__ float red[DSP][4][2];
  const int j = threadIdx.x, lane = j & 31, warp = j >> 5;
  const int g0 = blockIdx.x * DSP, X = a.X;
  const size_t P = size_t(a.P);
  if (j < DSP * 2) {
    const int p = j >> 1, gi = min(g0 + p, a.P - 1);
    zz[p][j & 1] = a.z[2 * size_t(gi) + (j & 1)];
  }
  if (blockIdx.x == 0 && j == 0 && !packed_header_ok(a.packed, a.K_total, X))
    atomicOr(a.status, unsigned(VLG_STATUS_BAD_PACKED));
  float (*dxs)[XP] = reinterpret_cast<float (*)[XP]>(&h2[0][0]);
  float dzacc = 0.f;   // backward, thread t < 64: component t & 1 of point t >> 1
  bool bad = j < DSP * 2 && g0 + (j >> 1) < a.P && !finite32(a.z[2 * size_t(g0) + j]);   // as in tc_decode_kernel
  // expected energy: thread j < X sums ||x_k - mu_t||^2 of column j for each point; point p = t * N + n of its curve
  const int T = EXPECT ? a.P / a.N : 0;
  const size_t nbr = size_t(a.N) * size_t(X);
  float vacc[EXPECT ? DSP : 1];
#pragma unroll
  for (int p = 0; p < (EXPECT ? DSP : 1); ++p) vacc[p] = 0.f;
  __syncthreads();
  for (int k = 0; k < a.K; ++k) {
    const float* d = dec_ptr(a.packed, k);
    uint32_t m1 = 0, m2 = 0;
    {
      const float wa = d[OFF_W1X + j], wb = d[OFF_W1Y + j], bb = d[OFF_B1 + j];
#pragma unroll
      for (int p = 0; p < DSP; ++p) {
        const float pre = fmaf(wb, zz[p][1], fmaf(wa, zz[p][0], bb));
        if (pre > 0.f) m1 |= 1u << p;
        h1[p][j] = fmaxf(pre, 0.f);
      }
    }
    __syncthreads();
    {
      float acc[DSP];
      const float bb = d[OFF_B2 + j];
#pragma unroll
      for (int p = 0; p < DSP; ++p) acc[p] = bb;
      for (int i = 0; i < H; ++i) {
        const float w = __ldg(d + OFF_W2T + i * H + j);
#pragma unroll
        for (int p = 0; p < DSP; ++p) acc[p] = fmaf(h1[p][i], w, acc[p]);
      }
      if (!BWD) {
#pragma unroll
        for (int p = 0; p < DSP; ++p) h2[p][j] = fmaxf(acc[p], 0.f);
      }
      if (BWD || EGRAD) {
#pragma unroll
        for (int p = 0; p < DSP; ++p)
          if (acc[p] > 0.f) m2 |= 1u << p;
      }
    }
    if (!BWD) {
      float gk[EGRAD ? DSP : 1];   // EnergyGrad: column j of the dE/dx rows, up to the factor 2 / K
      __syncthreads();
      if (j < X) {
        float acc[DSP];
        const float bb = d[OFF_B3 + j];
#pragma unroll
        for (int p = 0; p < DSP; ++p) acc[p] = bb;
        for (int i = 0; i < H; ++i) {
          const float w = __ldg(d + OFF_W3T + i * XP + j);
#pragma unroll
          for (int p = 0; p < DSP; ++p) acc[p] = fmaf(h2[p][i], w, acc[p]);
        }
        if (MODE == DecodeMode::Forward) {
#pragma unroll
          for (int p = 0; p < DSP; ++p)
            if (g0 + p < a.P) {
              a.x[(size_t(k) * P + size_t(g0 + p)) * size_t(X) + j] = acc[p];
              bad |= !finite32(acc[p]);
            }
        } else if (MODE == DecodeMode::Mean) {
#pragma unroll
          for (int p = 0; p < DSP; ++p)
            if (g0 + p < a.P) {
              float* m = a.mu + size_t(g0 + p) * size_t(X) + j;
              const float s = k == 0 ? acc[p] : *m + acc[p];
              *m = k == a.K - 1 ? s / float(a.K) : s;
              if (k == a.K - 1) bad |= !finite32(s);
            }
        } else {
#pragma unroll
          for (int p = 0; p < DSP; ++p) {
            if (EGRAD) gk[p] = 0.f;
            if (g0 + p < a.P) {
              const int t = (g0 + p) / a.N;
              const float* m0 = a.mu + size_t(g0 + p) * size_t(X) + j;
              const float* m1 = t > 0 ? m0 - nbr : m0 + nbr;
              const float dm = acc[p] - __ldg(m0);
              vacc[p] = fmaf(dm, dm, vacc[p]);
              if (EGRAD)
                gk[p] = t > 0 && t < T - 1 ? (acc[p] - __ldg(m1)) + (acc[p] - __ldg(m0 + nbr)) : acc[p] - __ldg(m1);
            }
          }
        }
      }
      __syncthreads();
      if (!EGRAD) continue;
      // (h2 is read by every thread above: its rows now take the dE/dx rows)
      if (j < X)
#pragma unroll
        for (int p = 0; p < DSP; ++p) dxs[p][j] = gk[p];
    } else {
      // backward: dx rows of this decoder
      for (int i = j; i < DSP * XP; i += 128) {
        const int p = i / XP, o = i - p * XP;
        dxs[p][o] = (o < X && g0 + p < a.P) ? a.dx[(size_t(k) * P + size_t(g0 + p)) * size_t(X) + o] : 0.f;
      }
    }
    __syncthreads();   // h1 is read by every thread above; dxs is complete
    {
      float acc[DSP];   // dh2 of unit j = m2 . (dx W3)[j]
#pragma unroll
      for (int p = 0; p < DSP; ++p) acc[p] = 0.f;
      for (int o = 0; o < X; ++o) {
        const float w = __ldg(d + OFF_W3 + o * H + j);
#pragma unroll
        for (int p = 0; p < DSP; ++p) acc[p] = fmaf(dxs[p][o], w, acc[p]);
      }
#pragma unroll
      for (int p = 0; p < DSP; ++p) h1[p][j] = ((m2 >> p) & 1u) ? acc[p] : 0.f;
    }
    __syncthreads();
    {
      float acc[DSP];   // dh1 of unit j = m1 . (dh2 W2)[j]
#pragma unroll
      for (int p = 0; p < DSP; ++p) acc[p] = 0.f;
      for (int i = 0; i < H; ++i) {
        const float w = __ldg(d + OFF_W2 + i * H + j);
#pragma unroll
        for (int p = 0; p < DSP; ++p) acc[p] = fmaf(h1[p][i], w, acc[p]);
      }
      const float wa = d[OFF_W1X + j], wb = d[OFF_W1Y + j];
#pragma unroll
      for (int p = 0; p < DSP; ++p) {
        const float dh = ((m1 >> p) & 1u) ? acc[p] : 0.f;
        const float cx = warp_sum(dh * wa), cy = warp_sum(dh * wb);
        if (lane == 0) { red[p][warp][0] = cx; red[p][warp][1] = cy; }
      }
    }
    __syncthreads();
    if (j < 2 * DSP) {
      const int p = j >> 1, c = j & 1;
      dzacc += (red[p][0][c] + red[p][1][c]) + (red[p][2][c] + red[p][3][c]);
    }
    // (the next decoder writes h1 and red only after two more barriers)
  }
  if ((BWD || EGRAD) && j < 2 * DSP && g0 + (j >> 1) < a.P) {
    const float g = EGRAD ? 2.f * dzacc / float(a.K) : dzacc;
    a.dz[2 * size_t(g0) + j] = g;
    bad |= !finite32(g);
  }
  if (EXPECT) {
    // e_t = c_t V_t + ||mu_{t+1} - mu_t||^2: both sums over the columns j < X, across the block
    __syncthreads();   // (EnergyGrad: red was read above)
#pragma unroll
    for (int p = 0; p < DSP; ++p) {
      const int gp = min(g0 + p, a.P - 1), t = gp / a.N;
      float dd = 0.f;
      if (j < X && t < T - 1) {
        const float dm = __ldg(a.mu + size_t(gp) * size_t(X) + nbr + j) - __ldg(a.mu + size_t(gp) * size_t(X) + j);
        dd = dm * dm;
      }
      const float v = warp_sum(j < X ? vacc[p] : 0.f), s = warp_sum(dd);
      if (lane == 0) { red[p][warp][0] = v; red[p][warp][1] = s; }
    }
    __syncthreads();
    if (j < DSP && g0 + j < a.P) {
      const int t = (g0 + j) / a.N;
      const float v = (red[j][0][0] + red[j][1][0]) + (red[j][2][0] + red[j][3][0]);
      const float s = (red[j][0][1] + red[j][1][1]) + (red[j][2][1] + red[j][3][1]);
      const float et = float(int(t > 0) + int(t < T - 1)) * (v / float(a.K)) + s;
      a.e[g0 + j] = et;
      bad |= !finite32(et);
    }
  }
  if (bad) atomicOr(a.status, unsigned(VLG_STATUS_NONFINITE));
}

// E_n = sum_t e[t * N + n] in increasing t: one thread per curve, no atomics
__global__ void curve_sum_kernel(const float* e, int N, int T, float* energy, unsigned int* status) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float s = 0.f;
  for (int t = 0; t < T; ++t) s += e[size_t(t) * size_t(N) + n];
  energy[n] = s;
  if (!finite32(s)) atomicOr(status, unsigned(VLG_STATUS_NONFINITE));
}

}  // namespace

// One launch of the decode kernel of MODE in the kernel format of `precision`.
template <DecodeMode MODE>
cudaError_t launch_mode(const DecodeArgs& a, int precision, cudaStream_t stream) {
  constexpr bool DX = MODE == DecodeMode::Backward || MODE == DecodeMode::EnergyGrad;   // runs B3, B2
  if (precision == VLG_PRECISION_FP32) {
    const int blocks = (a.P + DSP - 1) / DSP;
    simt_decode_kernel<MODE><<<blocks, 128, 0, stream>>>(a);
    return cudaGetLastError();
  }
  const int ntiles = (a.P + 127) / 128;
  const int grid = ntiles < DEC_CTAS_PER_SM * persistent_grid(ntiles) ? ntiles : DEC_CTAS_PER_SM * persistent_grid(ntiles);
  auto launch = [&](auto kernel) -> cudaError_t {
    cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(DEC_SMEM));
    if (err != cudaSuccess) return err;
    kernel<<<grid, DEC_THREADS, DEC_SMEM, stream>>>(a);
    return cudaGetLastError();
  };
  switch (precision) {
    case VLG_PRECISION_TF32: return launch(tc_decode_kernel<FMT_TF32, MODE>);
    case VLG_PRECISION_F16: return launch(tc_decode_kernel<FMT_F16, MODE>);
    case VLG_PRECISION_F16X3F:
      if constexpr (DX) return launch(tc_decode_kernel<FMT_F16X3F, MODE>);
      else return launch(tc_decode_kernel<FMT_F16X3, MODE>);   // no backward GEMMs: the mixed format is the 3-term format
    default: return launch(tc_decode_kernel<FMT_F16X3, MODE>);
  }
}

cudaError_t launch_decode(const void* packed, int K_total, int X, int K, int P, const float* z, const float* dx, float* x,
                          float* dz, int precision, void* workspace, cudaStream_t stream) {
  DecodeArgs a{packed, K_total, X, K, P, z, dx, x, dz, static_cast<unsigned int*>(workspace) + 1, 0, nullptr, nullptr};
  cudaError_t e = cudaMemsetAsync(workspace, 0, VLG_DECODE_WORKSPACE_BYTES, stream);
  if (e != cudaSuccess) return e;
  return dz ? launch_mode<DecodeMode::Backward>(a, precision, stream) : launch_mode<DecodeMode::Forward>(a, precision, stream);
}

cudaError_t launch_expected_energy(const void* packed, int K_total, int X, int K, int N, int T, const float* z,
                                   float* energy, float* grad_z, int precision, void* workspace, cudaStream_t stream) {
  const size_t P = size_t(T) * size_t(N);
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  float* mu = reinterpret_cast<float*>(ws + VLG_DECODE_WORKSPACE_BYTES);
  float* e_t = mu + P * size_t(X);
  unsigned int* status = reinterpret_cast<unsigned int*>(ws) + 1;
  DecodeArgs a{packed, K_total, X, K, int(P), z, nullptr, nullptr, grad_z, status, N, mu, e_t};
  cudaError_t err = cudaMemsetAsync(workspace, 0, VLG_DECODE_WORKSPACE_BYTES, stream);
  if (err == cudaSuccess) err = launch_mode<DecodeMode::Mean>(a, precision, stream);
  if (err == cudaSuccess)
    err = grad_z ? launch_mode<DecodeMode::EnergyGrad>(a, precision, stream) : launch_mode<DecodeMode::Energy>(a, precision, stream);
  if (err != cudaSuccess) return err;
  curve_sum_kernel<<<(N + 127) / 128, 128, 0, stream>>>(e_t, N, T, energy, status);
  return cudaGetLastError();
}

}  // namespace vlg
