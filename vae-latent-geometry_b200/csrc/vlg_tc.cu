// tcgen05 geodesic step kernel -- the tensor-core variants.
//
// Persistent CTAs (one per SM, 640 threads) pull work units -- (curve, chunk of Adam steps) -- from
// a global queue; a curve's chunks are chained through its omega/m/v in HBM, so a launch of
// `steps` steps has no tail longer than one chunk.  The two 128-wide decoder layers and their
// transposes run as tcgen05.mma with
//   * M = 128 rows = the 128 TMEM lanes,
//   * the A operand (activations) living in TENSOR MEMORY: the epilogue threads write the
//     next layer's input with tcgen05.st after reading the accumulator with tcgen05.ld,
//   * the B operand (weights) streamed from L2 into per-chain shared-memory rings by the TMA
//     engine (1-D bulk copies of pre-packed no-swizzle K-major images, mbarrier complete_tx),
//   * fp32 accumulators in TMEM.
// Three operand formats (template parameter FMT, VLG_PRECISION_*):
//   FMT_TF32   kind::tf32, operands rounded to TF32 (<= 1e-3 relative on lengths)
//   FMT_F16    kind::f16, fp16 operands: same 11-bit significand, half the MMAs and weight bytes
//   FMT_F16X3  kind::f16, every operand as hi + lo fp16 pairs, three MMAs per product: fp32-grade
//   FMT_F16X3F the same in the forward GEMMs (energies fp32-grade), single-term fp16 in the backward GEMMs
//
// ROW COMPACTION.  The MC energy touches, per curve point, only the decoders drawn for the two
// segments that meet there (<= 2M of K; 3.4 of 10 on average), and the reference's dense
// K x T forward/backward spends two thirds of its FLOPs on outputs that are multiplied by zero.
// Here a curve is cut into windows of W points (W chosen on the host so that a decoder is drawn by
// ~115 points of a window on average; W-1 segments); for every decoder the points
// of the window that drew it are gathered into the rows of one 128-row MMA tile ("item"; a
// decoder drawn by more than 128 points simply gets several items).  Results are identical:
// each selected (point, decoder) pair goes through exactly the same arithmetic.
//
// Warp roles: warps 0/1 = weight producers of chain 0/1 (one lane each), warp 2 = MMA issuer
// (all lanes run the loop, one elected lane's instructions take effect), warps 3-10 and 11-18 = two
// epilogue groups of 8 warps, warp 19 = window setup.  Each group owns a "chain"
// of 256 TMEM columns and every other item.  The MMA issuer serves whichever chain has its
// operand ready, which is why every chain has its own weight ring.  Inside a group two threads
// share a row (TMEM lane) and split its columns: four epilogue warps per scheduler hide TMEM /
// shared-memory latency.
//
// Per window, one window ahead in the setup warp: draws (one word per point: the decoders of the <= 4 segment ends
// that meet there) -> per-decoder row lists in point order (deterministic item membership) -> item list; all of it
// double buffered by window parity.  Then in the epilogue: points of the window ->
// forward items (layer 1 on CUDA cores, exact fp32) -> selected outputs stored
// with plain stores, one writer per slot (left-end output x1 of a segment in shared memory,
// right-end output x2 in an L2-resident workspace) -> one pass forms x2-x1 and the energy ->
// backward items (input gradient only; layer-2 ReLU masks as bits in the workspace, layer-1
// mask recomputed) -> dz per (point, draw slot) cell -> d(omega).  Penalty gradient and Adam as in vlg_simt.cu.
//
// Where the time goes (VLG_TC_STATS build, per 128-row item of a chain, 3-term mode): 43 % epilogue phases
// (7 per item, latency bound: two warps of a group per scheduler), 40 % waiting for the four GEMMs (a third of
// it the MMAs themselves, the rest issue / commit / wake-up latency and the other chain's MMAs), 16 % per-window
// phases (the x2-x1 pass: bandwidth of a 119 KB buffer, d(omega); in these round-2 figures also the row lists, which
// the setup warp now builds off the chains).  Tensor memory holds two chains, which is what bounds the overlap; see DESIGN.md 4.4 for the experiments that did not help.
#include <cuda_fp16.h>
#include <stdlib.h>

#include <type_traits>

#include "../../include/vlg.h"
#include "vlg_common.cuh"
#include "vlg_kernels.h"
#include "vlg_tcgen05.cuh"

namespace vlg {

#ifdef VLG_TC_STATS
// debug build only: per-CTA wait-cycle counters [cta][8]
__device__ long long g_tc_stats[1024 * 8];
#define STAT_T0() long long _t0 = clock64()
#define STAT_ADD(var) var += clock64() - _t0
// per-phase cycle accounting of the first warp of each epilogue group: [cta][chain][24]
__device__ long long g_tc_phase[1024 * 48];
#define PH_DECL() volatile long long ph_[24]; long long ph_t_ = clock64(); for (int i_ = 0; i_ < 24; ++i_) ph_[i_] = 0
#define PH(i) do { if (tg == 0) { const long long n_ = clock64(); ph_[i] += n_ - ph_t_; ph_t_ = n_; } } while (0)
// arrival skew inside a group: every epilogue warp notes when it arrived, the first warp of the group sees after the
// round trip how much later the last one came
#define ARR() do { if (lane == 0) arr_t_[ew] = clock64(); } while (0)
#define SKEW(i) do { if (tg == 0) { long long mx_ = 0; for (int w_ = 0; w_ < 8; ++w_) mx_ = max(mx_, arr_t_[chain_id * 8 + w_]); \
  if (VLG_TC_STATS_SKEW) { ph_[i] += mx_ - arr_t_[ew]; ph_[21] += iss_t_[2 * chain_id] - mx_; ph_[22] += iss_t_[2 * chain_id + 1] - iss_t_[2 * chain_id]; ph_[23] += clock64() - iss_t_[2 * chain_id + 1]; } } } while (0)
#ifndef VLG_TC_STATS_SKEW
#define VLG_TC_STATS_SKEW 0   // 1: slots 17..23 = arrival skew / issuer timeline; 0: sub-phases of the per-window work
#endif
#define PHW(i) do { if (!VLG_TC_STATS_SKEW) PH(i); } while (0)
#define PH_FLUSH() do { if (tg == 0 && blockIdx.x < 1024) for (int i_ = 0; i_ < 24; ++i_) g_tc_phase[(blockIdx.x * 2 + chain_id) * 24 + i_] = ph_[i_]; } while (0)
#else
#define STAT_T0()
#define STAT_ADD(var)
#define PH_DECL()
#define PH(i)
#define ARR()
#define SKEW(i)
#define PHW(i)
#define PH_FLUSH()
#endif

namespace {

using namespace tc;

#ifndef VLG_TC_TILE_TB
#define VLG_TC_TILE_TB 4              // dE/dx tile pass (multi-curve windows): tasks in flight per thread
#endif
#ifndef VLG_TC_G_AHEAD
#define VLG_TC_G_AHEAD 1               // single-term backward: next item's dE/dx rows built under the current B2
#endif
constexpr int TC_THREADS = 640;       // 3 control warps + 16 epilogue warps + the window-setup warp
constexpr int GROUP_THREADS = 256;    // one epilogue group (chain)
constexpr int EPI_THREADS = 512;
constexpr int FIRST_EPI_WARP = 3;
constexpr int SETUP_WARP = FIRST_EPI_WARP + 16;
constexpr int STAGE_BYTES = 16384;
constexpr int MAX_STAGES = 5;         // per chain
constexpr int XD_STRIDE = 52;         // floats per stored decoder output row (X <= 52; 16 B rows)
constexpr int GT_BYTES = 32768;       // dE/dx operand tile of one item in the workspace: fp16 16 KB (3-term: hi tile + lo tile),
                                      // tf32 32 KB; canonical no-swizzle K-major image [k-chunk][row][16 B], like the weights
constexpr int TC_MAX_W = 512;         // points per window, one curve per window (neighbouring windows share one point)
constexpr int TC_MAX_WG = 2048;       // points per window when it holds several whole curves (XL2 kernels)
constexpr int TC_MAX_G = 8;           // curves per window (XL2 kernels)
constexpr int OM_STRIDE = 6 * MAX_KB + 2;   // per-curve omega | adam m | adam v
constexpr int TC_MAX_M = 2;           // MC samples per block (any number of samples: blocks of two)
constexpr int TC_MAX_K = 128;         // decoders
constexpr int MAX_ITEMS = TC_MAX_K + 2 * TC_MAX_M * TC_MAX_WG / 128 + 8;  // sum_k ceil(n_k/128) <= K + 2*M*W/128

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
// 0xFFFF in every 16-bit half of `w` that holds a positive fp16 value (one HSET2.BM)
__device__ __forceinline__ uint32_t pos_mask_h2(uint32_t w) {
  return __hgt2_mask(*reinterpret_cast<const __half2*>(&w), __float2half2_rn(0.f));
}
// ReLU-mask word layouts.  MASKH (fp16 single-term kernel only): pair p = elements (2p, 2p+1) of a 32-column
// tile -> bits p and 16+p, taken straight from the packed fp16 activations (HSET2 + LOP3 per pair instead of
// 2 x (FSETP + LOP)); expanded in the backward pass to 16-bit lane masks with one IMAD.
// Backward quantities (dE/dx and the hidden-layer gradients) are scaled by 2^6 before they are rounded to
// fp16 and unscaled in fp32 when dz is accumulated: gradients of a converged curve are O(1e-2 .. 1e-5)
// per element, fp16 loses precision below 6e-5.
constexpr float F16_GRAD_SCALE = 64.f;

// round-to-nearest to TF32 for finite values: the tensor core ignores the 13 low mantissa bits
__device__ __forceinline__ uint32_t tf32_round_bits(uint32_t b) { return b + 0x1000u; }
// relu, then TF32 round-to-nearest on the bit pattern.  (An integer-max formulation,
// max(int(bits + 0x1000), 0), produced wrong results when combined with the packed f32x2
// intrinsics under nvcc 12.9 -- keep the float max.)
__device__ __forceinline__ uint32_t relu_tf32(float v) { return __float_as_uint(fmaxf(v, 0.f)) + 0x1000u; }

// 0xFF in byte j iff draw slot j of point pt holds decoder k (TcSmem::sel: one word per point)
__device__ __forceinline__ uint32_t slot_match(const uint8_t* sel, int pt, int k) {
  return __vcmpeq4(reinterpret_cast<const uint32_t*>(sel)[pt], uint32_t(k) * 0x01010101u);
}
// "operand ready" of an epilogue group: every thread has completed and fenced its tensor-memory stores; one arrival
// per warp (the mbarrier counts the group's 8 warps) instead of 256 serialized arrivals on one shared-memory word
__device__ __forceinline__ void group_arrive(uint64_t* bar, int lane) {
  __syncwarp();
  if (lane == 0) mbar_arrive(bar);
}
__device__ __forceinline__ void named_bar(int id, int count) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_elect(uint64_t* bar, uint32_t leader) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t"
      "setp.ne.b32 q, %1, 0;\n\t"
      "@q mbarrier.arrive.shared::cta.b64 _, [%0];\n\t}" ::"r"(smem_u32(bar)), "r"(leader)
      : "memory");
}
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}

// work-queue header at the start of the workspace: 64 words ([0] next unit, [1] status flags VLG_STATUS_*)
// + one progress word per curve, 256 B aligned
__host__ __device__ inline size_t tc_queue_words(int N) { return (size_t(64 + N) + 63) / 64 * 64; }

// Per-CTA slice of the L2-resident workspace, in 32-bit words: layer-2 ReLU masks [items][128 rows][4],
// left-end decoder outputs x1 [M][W][52] and right-end outputs x2 [M][W][52] (fp32), dE/dx operand tiles
// [items][GT_BYTES]; items = tc_max_items >= sum_k ceil(n_k / 128).
__host__ __device__ inline int tc_max_items(int K, int M, int W) { return K + 2 * M * W / 128 + 2; }
__host__ __device__ inline size_t tc_ws_cta_words(int K, int M, int W) {
  const size_t items = size_t(tc_max_items(K, M, W));
  return (items * 512 + 2 * size_t(M) * W * XD_STRIDE + items * (GT_BYTES / 4) + 31) / 32 * 32;
}

struct WinCtl {
  int nitems;    // < 0: no more work units
  int base;      // first decoder of the curve's weight set inside `packed` (StepParams::dec_base)
  unsigned int unit;   // work unit the window belongs to (>= total units: no more work)
  uint16_t item[MAX_ITEMS];  // decoder | pass << 8
};

// Wait for the chain's accumulator: every lane polls the mbarrier (lane 0 polling + __syncwarp: measured -5 %).
__device__ __forceinline__ void acc_wait(uint64_t* bar, uint32_t parity, int lane) {
  (void)lane;
  mbar_wait(bar, parity);
}

struct TcSmem {
  unsigned char* ring;  // [chain][stage] 16 KB
  float* XD;            // [m][W][52] left-end outputs x1, then x2 - x1 (only when they fit: XL2 == 0; else in the workspace)
  // sel, rows, crow and ctl are written by the window-setup warp one window ahead: double buffered by window parity
  uint8_t* sel;         // [2][tc_sel_words(W)][4] per POINT: the decoders drawn for the segments that meet there -- byte 2m: left
                        // end of its own segment (MC sample m), byte 2m+1: right end of the previous one; 255: none (also every
                        // byte of the words from W on).  One 32-bit load per row.
  uint16_t* rows;       // [2][2 M W] points of the window that drew decoder k, in increasing point order: rows[roff[k] .. + cnt[k])
  uint32_t* crow;       // [2][TC_MAX_K] roff[k] | cnt[k] << 16
  WinCtl* ctl;          // [2] item lists
  float* sw;            // [chain][SW_SLOTS] 576 floats: W1 (planar), b1, b2, b3 of an item's decoder
  float2* zs;           // W latent points of the window
  float2* dzs;          // [4][W]: dz of point pt from the decoder of its draw slot (m0 left, m0 right, m1 left, m1 right)
  float* coef;          // [G][64]
  float* basis;         // 288
  float* om;            // [G][OM_STRIDE]
  float* gacc;          // [G][20]
  float* pab;           // [G][4] end points a, b
  float* etot;          // [G][2] energy / length of the step so far
  float* red;           // [16][20] d(omega) partials per warp, then [G][32] energy | length partials per warp
  float2* dzx;          // [chain][half][128] dz partial of a row's two half-threads (last backward item of the chain)
  uint64_t* bars;       // full[2][MAX_STAGES], empty[2][MAX_STAGES], a_ready[2], acc_ready[2], win_ready[2], sw_full[2][SW_SLOTS], ctl_free[2], g_ready
  uint32_t* tmem_base;  // [0] TMEM base address
};

constexpr int CTL_FLOATS = (2 * sizeof(WinCtl) + 3) / 4;
constexpr int SW_SLOTS = 4;            // small-weight buffers per chain (see the producer)
constexpr int BAR_WORDS = 2 * (4 * MAX_STAGES + 6 + 2 * SW_SLOTS + 3);
static_assert(TC_MAX_M == 2, "the row-list build tests four candidates per point");

// Fixed-size pieces first, at compile-time offsets from the start of dynamic shared memory (their
// addresses fold into immediates -- the epilogue code is short of registers), then the window-sized
// arrays, then the weight rings.  GM = curves per window the kernel is built for (1, or TC_MAX_G for XL2).
template <int GM>
struct Fix {
  static constexpr int SW = 0;                                   // 2 chains x SW_SLOTS x 576
  static constexpr int COEF = SW + 2 * SW_SLOTS * 576;           // GM x 64
  static constexpr int BASIS = COEF + GM * 64;                   // 4 * MAX_NPOLY * MAX_KB
  static constexpr int OM = BASIS + 4 * MAX_NPOLY * MAX_KB;      // GM x OM_STRIDE
  static constexpr int GACC = OM + GM * OM_STRIDE;               // GM x 20
  static constexpr int PAB = GACC + GM * 20;                     // GM x 4
  static constexpr int ETOT = PAB + GM * 4;                      // GM x 2
  static constexpr int RED = ETOT + GM * 2;                      // 320 + GM x 32
  static constexpr int DZX = (RED + 320 + GM * 32 + 1) / 2 * 2;  // 2 x 2 x 128 float2
  static constexpr int BARS = DZX + 1024;                         // BAR_WORDS (8-byte aligned)
  static constexpr int TMEM = BARS + BAR_WORDS;                  // 4
  static constexpr int CTL = TMEM + 4;                           // CTL_FLOATS
  static constexpr int CROW = CTL + CTL_FLOATS;                  // 2 x TC_MAX_K
  static constexpr int FLOATS = (CROW + 2 * TC_MAX_K + 3) / 4 * 4;   // XD starts 16-byte aligned
};

__host__ __device__ inline int tc_chunks(int W) { return (W + 511) / 512; }
// one buffer of TcSmem::sel: W + 1 words, rounded up to whole 16-byte loads
__host__ __device__ inline int tc_sel_words(int W) { return (W + 1 + 3) / 4 * 4; }

template <int GM>
__device__ __forceinline__ TcSmem tc_carve(unsigned char* base, int W, int K, int M, bool xd_in_smem) {
  using FX = Fix<GM>;
  TcSmem s;
  float* f = reinterpret_cast<float*>(base);
  s.sw = f + FX::SW;
  s.coef = f + FX::COEF;
  s.basis = f + FX::BASIS;
  s.om = f + FX::OM;
  s.gacc = f + FX::GACC;
  s.pab = f + FX::PAB;
  s.etot = f + FX::ETOT;
  s.red = f + FX::RED;
  s.dzx = reinterpret_cast<float2*>(f + FX::DZX);
  s.bars = reinterpret_cast<uint64_t*>(f + FX::BARS);
  s.tmem_base = reinterpret_cast<uint32_t*>(f + FX::TMEM);
  s.ctl = reinterpret_cast<WinCtl*>(f + FX::CTL);
  s.crow = reinterpret_cast<uint32_t*>(f + FX::CROW);
  f += FX::FLOATS;
  s.XD = f; f += xd_in_smem ? M * W * XD_STRIDE : 0;
  s.sel = reinterpret_cast<uint8_t*>(f); f += 2 * tc_sel_words(W);   // 16-byte aligned (read as uint4 by the setup warp)
  s.zs = reinterpret_cast<float2*>(f); f += 2 * W;
  s.dzs = reinterpret_cast<float2*>(f); f += 2 * 4 * W;
  s.rows = reinterpret_cast<uint16_t*>(f);
  const size_t ring_off = (size_t(reinterpret_cast<unsigned char*>(f) - base) + 2 * size_t(2 * M) * W * 2 + 127) / 128 * 128;
  s.ring = base + ring_off;
  return s;
}

}  // namespace

static size_t tc_smem_fixed_bytes(int W, int K, int M, int xl2) {
  // everything but the weight rings, in the order of tc_carve (+ alignment slack before the rings)
  const size_t fix = xl2 ? Fix<TC_MAX_G>::FLOATS : Fix<1>::FLOATS;
  size_t fl = fix + (xl2 ? 0 : size_t(M) * W * XD_STRIDE) + 2 * size_t(tc_sel_words(W)) + 2 * size_t(W) + 2 * 4 * size_t(W);
  return (fl * 4 + 2 * size_t(2 * M) * W * 2 + 127) / 128 * 128;
}
static int tc_stages(int W, int K, int M, int xl2) {
  const long budget = 232448 - long(tc_smem_fixed_bytes(W, K, M, xl2));
  long nst = budget / (2 * STAGE_BYTES);
  if (nst > MAX_STAGES) nst = MAX_STAGES;
  return int(nst);
}

template <StepMode MODE, int FMT, bool XL2>
__global__ void __launch_bounds__(TC_THREADS, 1) tc_curve_kernel(StepParams p, int nst, int W, int G_) {
  constexpr bool GRAD = MODE != StepMode::Energy;       // backward items
  constexpr bool GOUT = MODE == StepMode::EnergyGrad;   // gradient out instead of Adam
  constexpr bool xl2 = XL2;               // left-end outputs / differences in the L2 workspace instead of shared memory
  constexpr int GM = XL2 ? TC_MAX_G : 1;  // curves per window this kernel is built for
  const int G = XL2 ? G_ : 1;             // curves per window of this launch: G > 1 = G whole curves (W = G T points)
  const int Wp = W / G;                   // points of one curve in a window
  constexpr bool F16 = FMT != FMT_TF32;   // fp16 operands (one or two terms)
  constexpr bool X3F = FMT == FMT_F16X3 || FMT == FMT_F16X3F;   // 3-term split in the forward GEMMs (F2, F3)
  constexpr bool X3B = FMT == FMT_F16X3;                        // ... and in the backward GEMMs (B3, B2)
  extern __shared__ __align__(128) unsigned char smem_raw[];
#ifdef VLG_TC_STATS
  __shared__ volatile long long arr_t_[16];
  __shared__ volatile long long iss_t_[4];   // [chain]{seen ready, issued}
#endif
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // MC samples are processed two at a time ("sample blocks": one Philox call = the four draws of two samples, four draw
  // slots per point); M below is the capacity of a block, Mtot the number of samples the energy averages over
  const int Mtot = p.M, M = min(p.M, TC_MAX_M), K = p.K, T = p.T, n_poly = p.n_poly, Kb = p.Kb;
  TcSmem s = tc_carve<GM>(smem_raw, W, K, M, !xl2);
  const int WSEG = Wp - 1;  // segments of one curve per window
  uint64_t* full = s.bars;                       // [2][MAX_STAGES]
  uint64_t* empty = s.bars + 2 * MAX_STAGES;     // [2][MAX_STAGES]
  uint64_t* a_ready = s.bars + 4 * MAX_STAGES;
  uint64_t* acc_ready = s.bars + 4 * MAX_STAGES + 2;
  // window w's draws, row lists and item list are in buffer w & 1: win_ready[w & 1], phase w >> 1.  One barrier per
  // buffer: a waiter is never two phases behind, because buffer b is rewritten only after ctl_free[b]
  uint64_t* win_ready = s.bars + 4 * MAX_STAGES + 4;   // [2]
  uint64_t* sw_full = s.bars + 4 * MAX_STAGES + 6;   // [chain][SW_SLOTS]
  // buffer b may be rewritten once both producers, both chain states of the issuer and the epilogue are done with it
  uint64_t* ctl_free = s.bars + 4 * MAX_STAGES + 6 + 2 * SW_SLOTS;   // [2]
  // the dE/dx operand tiles of the window are in the workspace (phase = window)
  uint64_t* g_ready = s.bars + 4 * MAX_STAGES + 6 + 2 * SW_SLOTS + 2;
  const int nwin = (T - 1 + WSEG - 1) / WSEG;
  // work queue (zeroed by the host before the launch): [0] next unit, [64 + n] chunks done of curve n
  unsigned int* queue = reinterpret_cast<unsigned int*>(p.workspace);
  const int unit_steps = p.unit_steps;
  const int nchunks = (p.steps + unit_steps - 1) / unit_steps;
  const unsigned int ngroups = unsigned((p.N + G - 1) / G);   // work unit = (group of G consecutive curves, chunk of steps)
  const unsigned int total_units = ngroups * unsigned(nchunks);

  if (tid == 0) {
    for (int i = 0; i < 2 * MAX_STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(&a_ready[0], GROUP_THREADS / 32);   // one arrival per epilogue warp (group_arrive)
    mbar_init(&a_ready[1], GROUP_THREADS / 32);
    mbar_init(&acc_ready[0], 1);
    mbar_init(&acc_ready[1], 1);
    mbar_init(&win_ready[0], 1);
    mbar_init(&win_ready[1], 1);
    for (int i = 0; i < 2 * SW_SLOTS; ++i) mbar_init(&sw_full[i], 1);
    mbar_init(&ctl_free[0], 5);
    mbar_init(&ctl_free[1], 5);
    mbar_init(g_ready, 1);
    fence_mbar_init();
  }
  if (blockIdx.x == 0 && tid == 32 && !packed_header_ok(p.packed, p.K_total, p.X))
    atomicOr(&queue[1], unsigned(VLG_STATUS_BAD_PACKED));
  if (warp == 2) tmem_alloc(s.tmem_base, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *s.tmem_base;
  // Item i of a window (decoder k, rows 128q..128q+127 of k's row list) belongs to chain i & 1.
  // Per chain the tensor-core ops of a window are: for each of its items F2 F3, then (GRAD) for
  // each of its items B3 B2.  The item list of window w is published in ctl[w & 1] and
  // announced through win_ready[w & 1] (phase = w >> 1).
  if (warp < 2) {
    // ================= weight producer of chain `warp` (TMA bulk copies) =================
    if (lane == 0) {
      const int c = warp;
      uint64_t* fullc = full + c * MAX_STAGES;
      uint64_t* emptyc = empty + c * MAX_STAGES;
      unsigned char* ringc = s.ring + c * nst * STAGE_BYTES;
      int slot = 0;
      uint32_t ph = 0;
      unsigned swj = 0;   // stream index of the chain's items (forward and backward items of all windows)
      // dE/dx operand tiles of this CTA in the workspace (see the epilogue)
      const unsigned char* gtiles = reinterpret_cast<const unsigned char*>(
          reinterpret_cast<const uint32_t*>(p.workspace) + tc_queue_words(p.N) + size_t(blockIdx.x) * tc_ws_cta_words(K, M, W) +
          size_t(tc_max_items(K, M, W)) * 512 + 2 * size_t(M) * W * XD_STRIDE);
      for (long w = 0;; ++w) {
        mbar_wait(&win_ready[w & 1], uint32_t((w >> 1) & 1));
        const WinCtl* ctl = &s.ctl[w & 1];
        const int nit = ctl->nitems;
        if (nit < 0) break;  // no more work units
        bool g_seen = false;
        for (int phase = 0; phase < (GRAD ? 2 : 1); ++phase)
          for (int i = c; i < nit; i += 2) {
            const int k = ctl->base + (ctl->item[i] & 0xFF);
            // Small weights of this item into slot swj % SW_SLOTS.  No "slot free" barrier is needed: the
            // producer is here only after it issued every weight stage of the previous item, the last of
            // which went into a ring slot that an MMA of item j-1 or j-2 had released (the ring holds at
            // most 4 stages, an item has at least 3) -- so the epilogue threads, which all arrive before
            // an MMA is issued, are past item j-3, and slot j % 4 was last read by item j-4.
            {
              uint64_t* bar = &sw_full[c * SW_SLOTS + (swj % SW_SLOTS)];
              mbar_expect_tx(bar, 576 * 4);
              bulk_g2s(s.sw + (c * SW_SLOTS + (swj % SW_SLOTS)) * 576, dec_ptr(p.packed, k), 576 * 4, bar);
              ++swj;
            }
            for (int o = 0; o < 2; ++o) {
              const OpInfo oi = op_info<FMT>(phase * 2 + o);
              const char* src = reinterpret_cast<const char*>(dec_ptr(p.packed, k) + oi.img_off);
              const char* src_lo = reinterpret_cast<const char*>(dec_ptr(p.packed, k) + oi.img_lo);
              if (xl2 && phase == 1 && o == 0) {
                // B3: (weight stage, dE/dx tile stage) pairs in the order the issuer consumes them.  fp16: one pair,
                // the whole contraction (k < 64).  tf32 and 3-term: two pairs, one per half of the contraction
                // (tf32: 16 KB of each image per half; 3-term: hi half | lo half, 8 KB each, in one stage) -- so
                // no more than two stages are live at a time and a two-stage ring is enough.
                const char* gt = reinterpret_cast<const char*>(gtiles) + size_t(i) * GT_BYTES;
                constexpr int NPAIR = (F16 && !X3B) ? 1 : 2;
                for (int st = 0; st < 2 * NPAIR; ++st) {
                  const int kh = st >> 1;
                  const bool is_g = st & 1;
                  if (is_g && !g_seen) {   // the tiles of this window exist once the epilogue's pass is done
                    mbar_wait(g_ready, uint32_t(w & 1));
                    g_seen = true;
                  }
                  mbar_wait(&emptyc[slot], ph ^ 1);
                  mbar_expect_tx(&fullc[slot], STAGE_BYTES);
                  unsigned char* dst = ringc + slot * STAGE_BYTES;
                  if (X3B) {
                    const char* hi = is_g ? gt : src;
                    const char* lo = is_g ? gt + 16384 : src_lo;
                    bulk_g2s(dst, hi + kh * 8192, 8192, &fullc[slot]);
                    bulk_g2s(dst + 8192, lo + kh * 8192, 8192, &fullc[slot]);
                  } else {
                    bulk_g2s(dst, (is_g ? gt : src) + kh * STAGE_BYTES, STAGE_BYTES, &fullc[slot]);
                  }
                  if (++slot == nst) { slot = 0; ph ^= 1; }
                }
                continue;
              }
              // 3-term mode: the stages of the main image, then the stages of the residual image
              for (int st = 0; st < ((phase == 0 ? X3F : X3B) ? 2 : 1) * oi.nstages; ++st) {
                const char* from = st < oi.nstages ? src + size_t(st) * STAGE_BYTES : src_lo + size_t(st - oi.nstages) * STAGE_BYTES;
                mbar_wait(&emptyc[slot], ph ^ 1);
                mbar_expect_tx(&fullc[slot], STAGE_BYTES);
                bulk_g2s(ringc + slot * STAGE_BYTES, from, STAGE_BYTES, &fullc[slot]);
                if (++slot == nst) { slot = 0; ph ^= 1; }
              }
            }
          }
        mbar_arrive(&ctl_free[w & 1]);   // done reading this window's item list
      }
    }
  } else if (warp == 2) {
    // ================= MMA issuer: serves whichever chain is ready =================
    // The whole warp runs this loop convergently; one elected lane's tcgen05 instructions take effect.  (A second
    // issuer warp -- one per chain -- interleaves the chains' MMAs in the tensor pipe, "processor sharing": both
    // GEMMs finish late, and puts a fifth warp on one scheduler: measured no gain to -5 %, DESIGN.md 4.4.)
    {
      const uint32_t leader = elect_one();
      int slot[2] = {0, 0}, opi[2] = {0, 0}, nitc[2] = {0, 0};
      int ops_left[2] = {0, 0};      // ops of the chain's current window still to issue
      long win[2] = {0, 0};          // next window whose item list the chain has to pick up
      bool fin[2] = {false, false};
      uint32_t ph[2] = {0, 0}, ph_a[2] = {0, 0};
      long long w_full = 0, w_issue = 0;
      STAT_T0();
      bool served = true;
      while (!(fin[0] && fin[1])) {
        // (backing off with __nanosleep when nothing was ready: measured -1 % at 64 ns, -2 % at 200 ns)
        served = false;
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          if (fin[c]) continue;
          if (ops_left[c] == 0) {
            if (!mbar_test(&win_ready[win[c] & 1], uint32_t((win[c] >> 1) & 1))) continue;
            const int nit = s.ctl[win[c] & 1].nitems;
            if (nit < 0) { fin[c] = true; continue; }
            mbar_arrive_elect(&ctl_free[win[c] & 1], leader);   // the issuer only needs the item count
            nitc[c] = (nit - c + 1) / 2;  // items of this chain in the window
            ops_left[c] = nitc[c] * (GRAD ? 4 : 2);
            opi[c] = 0;
            ++win[c];
            if (ops_left[c] == 0) continue;
          }
          if (!mbar_test(&a_ready[c], ph_a[c])) continue;
          served = true;
          ph_a[c] ^= 1;
#ifdef VLG_TC_STATS
          if (lane == 0) iss_t_[2 * c] = clock64();
#endif
          tc_fence_after();
          // op order inside a window: F2 F3 per item, then B3 B2 per item
          const int optype = (opi[c] < 2 * nitc[c]) ? (opi[c] & 1) : 2 + ((opi[c] - 2 * nitc[c]) & 1);
          const OpInfo oi = op_info<FMT>(optype);
          const bool x3op = optype < 2 ? X3F : X3B;   // 3-term split of this GEMM
          const uint32_t idesc = F16 ? umma_idesc_f16(oi.n) : umma_idesc_tf32(oi.n, 0);
          const uint32_t chain = tmem + uint32_t(c) * 256u;
          uint64_t* fullc = full + c * MAX_STAGES;
          uint64_t* emptyc = empty + c * MAX_STAGES;
          const unsigned char* ringc = s.ring + c * nst * STAGE_BYTES;
          if (xl2 && optype == 2) {
            // B3 = dE/dx tile (A, shared memory) x W3 image (B, shared memory); (W, G) stage pairs as the producer
            // queued them.  Both images: K-major, 16-byte core-matrix rows, 128 rows per k-chunk (LBO 2048, SBO 128).
            constexpr int NPAIR = (F16 && !X3B) ? 1 : 2;
            const uint32_t dcol = chain + oi.d_col;
#pragma unroll
            for (int pr = 0; pr < NPAIR; ++pr) {
              const int s_w = slot[c];
              mbar_wait(&fullc[s_w], ph[c]);
              if (++slot[c] == nst) { slot[c] = 0; ph[c] ^= 1; }
              const int s_g = slot[c];
              mbar_wait(&fullc[s_g], ph[c]);
              if (++slot[c] == nst) { slot[c] = 0; ph[c] ^= 1; }
              tc_fence_after();
              const uint32_t wb = smem_u32(ringc + s_w * STAGE_BYTES), gb = smem_u32(ringc + s_g * STAGE_BYTES);
              if (!F16) {
#pragma unroll
                for (int ks = 0; ks < 4; ++ks)   // K = 8 per MMA: two k-chunks of 4 floats
                  umma_tf32_ss_elect(dcol, umma_smem_desc(gb + uint32_t(ks) * 4096u, 2048u, 128u),
                                     umma_smem_desc(wb + uint32_t(ks) * 4096u, 2048u, 128u), idesc, (pr | ks) ? 1u : 0u, leader);
              } else if (X3B) {
#pragma unroll
                for (int term = 0; term < 3; ++term) {   // Ghi Whi, Glo Whi, Ghi Wlo; lo halves sit 8 KB into the stage
                  const uint32_t a_s = gb + (term == 1 ? 8192u : 0u), b_s = wb + (term == 2 ? 8192u : 0u);
#pragma unroll
                  for (int ks = 0; ks < 2; ++ks)         // K = 16 per MMA: two k-chunks of 8 halves
                    umma_f16_ss_elect(dcol, umma_smem_desc(a_s + uint32_t(ks) * 4096u, 2048u, 128u),
                                      umma_smem_desc(b_s + uint32_t(ks) * 4096u, 2048u, 128u), idesc, (pr | term | ks) ? 1u : 0u, leader);
                }
              } else {
#pragma unroll
                for (int ks = 0; ks < 4; ++ks)
                  umma_f16_ss_elect(dcol, umma_smem_desc(gb + uint32_t(ks) * 4096u, 2048u, 128u),
                                    umma_smem_desc(wb + uint32_t(ks) * 4096u, 2048u, 128u), idesc, ks ? 1u : 0u, leader);
              }
              umma_commit_elect(&emptyc[s_w], leader);
              umma_commit_elect(&emptyc[s_g], leader);
            }
          } else
          for (int st = 0; st < (x3op ? 2 : 1) * oi.nstages; ++st) {
            if (!mbar_test(&fullc[slot[c]], ph[c])) { STAT_T0(); mbar_wait(&fullc[slot[c]], ph[c]); STAT_ADD(w_full); }
            tc_fence_after();
            const uint32_t sbase = smem_u32(ringc + slot[c] * STAGE_BYTES);
            const int nk = oi.nk;
            const bool w_lo = x3op && st >= oi.nstages;          // this stage holds residual weights
            const int kst = w_lo ? st - oi.nstages : st;       // which slice of the contraction
            {
              STAT_T0();
              // main weights: main operand (and, 3-term mode, the residual operand 64 columns up);
              // residual weights: main operand only
              for (int term = 0; term < ((x3op && !w_lo) ? 2 : 1); ++term)
                for (int ks = 0; ks < nk; ++ks) {
                  const uint64_t desc =
                      umma_smem_desc(sbase + uint32_t(ks) * 2u * uint32_t(oi.n) * 16u, uint32_t(oi.n) * 16u, 128u);
                  const uint32_t a_addr = chain + oi.a_col + uint32_t(term * 64) + uint32_t((kst * nk + ks) * 8);
                  const uint32_t accum = (st | ks | term) ? 1u : 0u;
                  if (F16)
                    umma_f16_ts_elect(chain + oi.d_col, a_addr, desc, idesc, accum, leader);
                  else
                    umma_tf32_ts_elect(chain + oi.d_col, a_addr, desc, idesc, accum, leader);
                }
              umma_commit_elect(&emptyc[slot[c]], leader);
              STAT_ADD(w_issue);
            }
            if (++slot[c] == nst) { slot[c] = 0; ph[c] ^= 1; }
          }
          umma_commit_elect(&acc_ready[c], leader);
#ifdef VLG_TC_STATS
          if (lane == 0) iss_t_[2 * c + 1] = clock64();
#endif
          ++opi[c];
          --ops_left[c];
        }
      }
#ifdef VLG_TC_STATS
      if (lane == 0 && blockIdx.x < 1024) {
        g_tc_stats[blockIdx.x * 8 + 2] = w_full;
        g_tc_stats[blockIdx.x * 8 + 3] = clock64() - _t0;
        g_tc_stats[blockIdx.x * 8 + 5] = w_issue;
      }
#endif
      (void)w_full; (void)w_issue;
    }
  } else if (warp < SETUP_WARP) {
    // ================= epilogue groups =================
    const int ew = warp - FIRST_EPI_WARP;       // 0..15
    const int chain_id = ew >> 3;               // group / chain
    const int half = (ew >> 2) & 1;             // which 64 of the 128 columns
    const int row = (warp & 3) * 32 + lane;     // TMEM lane = row of the item
    const int tg = half * 128 + row;            // 0..255 inside the group
    const int t512 = chain_id * 256 + tg;       // 0..511 over both groups
    const uint32_t lane_addr = uint32_t((warp & 3) * 32) << 16;
    const uint32_t chain = tmem + lane_addr + uint32_t(chain_id) * 256u;
    const uint32_t colX = chain, colY = chain + 128u;
    const int col0 = half * 64;                 // this thread's hidden units
    const int xc0 = half * 32;                  // this thread's output / G columns
    const int nq = half ? (XD_STRIDE - 32) / 4 : 8;  // float4 groups of this thread's output columns
    const int bar_id = 1 + chain_id;
    float* swbuf = s.sw + chain_id * SW_SLOTS * 576;
    unsigned swj = 0;                           // stream index of this chain's items, as in the producer
    uint32_t ph_acc = 0;
    const float coefm = 2.0f / float(Mtot);
    long long w_acc = 0;
    long wcount = 0;                            // windows processed by this CTA so far
    // this CTA's slice of the L2-resident workspace (tc_ws_cta_words): ReLU masks, both end-point outputs of
    // every segment, and the dE/dx operand tiles one fused pass builds from them for the backward items
    uint32_t* maskws = reinterpret_cast<uint32_t*>(p.workspace) + tc_queue_words(p.N) + size_t(blockIdx.x) * tc_ws_cta_words(K, M, W);
    float* X1g = reinterpret_cast<float*>(maskws + size_t(tc_max_items(K, M, W)) * 512);
    float* X1 = xl2 ? X1g : s.XD;   // left-end outputs, then the differences: shared memory when they fit
    float* X2 = X1g + size_t(M) * W * XD_STRIDE;
    unsigned char* Gt = reinterpret_cast<unsigned char*>(X2 + size_t(M) * W * XD_STRIDE);

    for (int i = t512; i < 4 * n_poly * Kb; i += EPI_THREADS) s.basis[i] = p.basis[i];
    PH_DECL();
    const int nchunk = XL2 ? tc_chunks(W) : 1;  // the window's points in chunks of 512 (thread = point)

    for (;;) {
      // ---- next work unit: (group of G curves n0 .. n0 + Gcur - 1, steps [step_lo, step_hi)) ----
      // The setup warp pulls it from the queue and names it in the item list of the unit's first window.
      mbar_wait(&win_ready[wcount & 1], uint32_t((wcount >> 1) & 1));
      const unsigned int unit = s.ctl[wcount & 1].unit;
      if (unit >= total_units) break;
      if (t512 == 0 && unit >= ngroups) {
        // a later chunk of a group: wait until its previous chunk has been written back
        const unsigned int* flag = &queue[64 + unit % ngroups];
        const unsigned int need = unit / ngroups;
        unsigned int have;
        do {
          asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(have) : "l"(flag) : "memory");
          if (have < need) __nanosleep(100);
        } while (have < need);
      }
      named_bar(3, EPI_THREADS);
      const int grp = int(unit % ngroups);
      const int n0 = grp * G, Gcur = XL2 ? min(G, p.N - n0) : 1;
      const int chunk = int(unit / ngroups);
      const int step_lo = chunk * unit_steps, step_hi = min(p.steps, step_lo + unit_steps);
      if (t512 < G * 2 * Kb) {
        const int j = t512 / (2 * Kb), c = t512 - j * 2 * Kb;
        if (j < Gcur) {
          const size_t o = size_t(n0 + j) * 2 * Kb + c;
          s.om[j * OM_STRIDE + c] = __ldcg(p.omega + o);
          if (MODE == StepMode::Optimize) {
            s.om[j * OM_STRIDE + 2 * MAX_KB + c] = __ldcg(p.adam_m + o);
            s.om[j * OM_STRIDE + 4 * MAX_KB + c] = __ldcg(p.adam_v + o);
          }
        } else {
          s.om[j * OM_STRIDE + c] = 0.f;
        }
      }
      if (t512 < 4 * G) {
        const int j = t512 >> 2, c = t512 & 3, n = n0 + min(j, Gcur - 1);
        s.pab[t512] = c < 2 ? p.a[2 * n + c] : p.b[2 * n + c - 2];
      }
      named_bar(3, EPI_THREADS);

      for (int step = step_lo; step < step_hi; ++step) {
        for (int idx = t512; idx < G * 8 * n_poly; idx += EPI_THREADS) {
          const int j = idx / (8 * n_poly), q = idx - j * 8 * n_poly;
          const int r = q >> 1, d = q & 1;
          float acc = 0.f;
          for (int k = 0; k < Kb; ++k) acc = fmaf(s.basis[r * Kb + k], s.om[j * OM_STRIDE + 2 * k + d], acc);
          s.coef[j * 64 + q] = acc;
        }
        if (t512 < G * 20) s.gacc[t512] = 0.f;
        // gradient-output mode: dE/da, dE/db of curve j accumulate in the Adam-moment slots of s.om, unused there
        if (GOUT && t512 < G * 4) s.om[(t512 >> 2) * OM_STRIDE + 2 * MAX_KB + (t512 & 3)] = 0.f;
        if (t512 < G * 2) s.etot[t512] = 0.f;
        named_bar(3, EPI_THREADS);
        PH(16);

        // one pass of the window body per (window, sample block): to the control warps a block is just another window
        for (int win = 0; win < nwin; ++win)
        for (int mb = 0; 2 * mb < Mtot; ++mb, ++wcount) {
          const int Mb = min(TC_MAX_M, Mtot - 2 * mb);   // samples of this block
          const int seg0 = win * WSEG;
          const int nseg = min(WSEG, T - 1 - seg0);   // segments of every curve in this window
          // ---- window setup: draws, row lists and item list from the setup warp; points and dz accumulators here ----
          const int buf = int(wcount & 1);
          mbar_wait(&win_ready[buf], uint32_t((wcount >> 1) & 1));
          const WinCtl* ctl = &s.ctl[buf];
          const uint8_t* sel = s.sel + size_t(buf) * tc_sel_words(W) * 4;
          const uint16_t* rows = s.rows + size_t(buf) * 2 * M * W;
          const uint32_t* crow = s.crow + buf * TC_MAX_K;
          for (int pt = t512; pt < W; pt += EPI_THREADS) {   // point pt = curve j = pt / Wp, local index i
            const int j = pt / Wp, i = pt - j * Wp;
            const float* ab = s.pab + 4 * j;
            s.zs[pt] = spline_point(p.t[min(seg0 + i, T - 1)], n_poly, s.coef + j * 64, make_float2(ab[0], ab[1]),
                                    make_float2(ab[2], ab[3]));
          }
          for (int i = t512; i < 4 * W; i += EPI_THREADS) s.dzs[i] = make_float2(0.f, 0.f);
          named_bar(3, EPI_THREADS);
          const int nitems = ctl->nitems;
          PH(6);
          // =============================== forward ===============================
          for (int it = chain_id; it < nitems; it += 2) {
            const int k = ctl->item[it] & 0xFF, q0 = (ctl->item[it] >> 8) * 128;
            const uint32_t cr = crow[k];
            const bool active = q0 + row < int(cr >> 16);
            // tcgen05.ld/st are warp-collective (.sync.aligned): a warp takes part as soon as one of
            // its 32 rows is in use; unused lanes compute on point 0 and store nothing
            const bool wact = q0 + (warp & 3) * 32 < int(cr >> 16);
            const int pt = active ? rows[(cr & 0xFFFFu) + q0 + row] : 0;
            // small weights of decoder k: loaded by the chain's producer (bulk copy -> mbarrier).  TF32
            // operands overwrite accumulators in place, so the group must also be done with the previous
            // item's D3 before layer 1 is stored; fp16 operands and accumulators never share columns.
            mbar_wait(&sw_full[chain_id * SW_SLOTS + (swj % SW_SLOTS)], (swj / SW_SLOTS) & 1u);
            if (!F16) named_bar(bar_id, GROUP_THREADS);
            const float* sw = swbuf + (swj % SW_SLOTS) * 576;
            ++swj;
            const float2 z = s.zs[pt];
            const float2 zx2 = make_float2(z.x, z.x), zy2 = make_float2(z.y, z.y);
            PH(0);
            // layer 1 (CUDA cores, fp32) -> A1 in X[col0 : col0+64]  (fp16: pairs in X[32 half : +32])
            if (F16) {
              if (wact) {
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {   // 32 hidden units = 16 packed columns per pass
                  uint32_t v[16], vl[16];
#pragma unroll
                  for (int j = 0; j < 32; j += 4) {
                    const int c = col0 + 32 * hh + j;
                    const float4 wx = *reinterpret_cast<const float4*>(sw + OFF_W1X + c);
                    const float4 wy = *reinterpret_cast<const float4*>(sw + OFF_W1Y + c);
                    const float4 bb = *reinterpret_cast<const float4*>(sw + OFF_B1 + c);
                    const float2 h0 = __ffma2_rn(make_float2(wy.x, wy.y), zy2,
                                                 __ffma2_rn(make_float2(wx.x, wx.y), zx2, make_float2(bb.x, bb.y)));
                    const float2 h1 = __ffma2_rn(make_float2(wy.z, wy.w), zy2,
                                                 __ffma2_rn(make_float2(wx.z, wx.w), zx2, make_float2(bb.z, bb.w)));
                    if (X3F) {
                      pack_hilo_h2(fmaxf(h0.x, 0.f), fmaxf(h0.y, 0.f), v[j >> 1], vl[j >> 1]);
                      pack_hilo_h2(fmaxf(h1.x, 0.f), fmaxf(h1.y, 0.f), v[(j >> 1) + 1], vl[(j >> 1) + 1]);
                    } else {
                      v[j >> 1] = pack_relu_h2(h0.x, h0.y);
                      v[(j >> 1) + 1] = pack_relu_h2(h1.x, h1.y);
                    }
                  }
                  tmem_st16(colX + half * 32 + 16 * hh, v);
                  if (X3F) tmem_st16(colX + 64 + half * 32 + 16 * hh, vl);
                }
              }
            } else if (wact) {
#pragma unroll
              for (int c0 = 0; c0 < 64; c0 += 32) {
                uint32_t v[32];
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                  const int c = col0 + c0 + j;
                  const float4 wx = *reinterpret_cast<const float4*>(sw + OFF_W1X + c);
                  const float4 wy = *reinterpret_cast<const float4*>(sw + OFF_W1Y + c);
                  const float4 bb = *reinterpret_cast<const float4*>(sw + OFF_B1 + c);
                  const float2 h0 = __ffma2_rn(make_float2(wy.x, wy.y), zy2,
                                               __ffma2_rn(make_float2(wx.x, wx.y), zx2, make_float2(bb.x, bb.y)));
                  const float2 h1 = __ffma2_rn(make_float2(wy.z, wy.w), zy2,
                                               __ffma2_rn(make_float2(wx.z, wx.w), zx2, make_float2(bb.z, bb.w)));
                  v[j] = relu_tf32(h0.x);
                  v[j + 1] = relu_tf32(h0.y);
                  v[j + 2] = relu_tf32(h1.x);
                  v[j + 3] = relu_tf32(h1.y);
                }
                tmem_st32(colX + col0 + c0, v);
              }
            }
            tmem_wait_st();
            tc_fence_before();
            ARR(); group_arrive(&a_ready[chain_id], lane);
            PH(1);
            // layer 2 epilogue: D2 (Y) -> relu(+b2) -> A2 (Y, in place), mask bits
            { STAT_T0(); acc_wait(&acc_ready[chain_id], ph_acc, lane); STAT_ADD(w_acc); }
            ph_acc ^= 1;
            tc_fence_after();
            PH(2); SKEW(17);
            if (wact) {
              // two passes of 32 columns: one live 32-register tile instead of two (no spills)
              uint32_t bits[2];
#pragma unroll
              for (int hh = 0; hh < 2; ++hh) {
                uint32_t v[32];
                uint32_t vlo[X3F ? 16 : 1];
                tmem_ld32_sync(colY + col0 + 32 * hh, v);
                uint32_t bb = 0;
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                  const float4 b0 = *reinterpret_cast<const float4*>(sw + OFF_B2 + col0 + 32 * hh + j);
                  const float2 p0 = __fadd2_rn(make_float2(__uint_as_float(v[j]), __uint_as_float(v[j + 1])), make_float2(b0.x, b0.y));
                  const float2 p1 = __fadd2_rn(make_float2(__uint_as_float(v[j + 2]), __uint_as_float(v[j + 3])), make_float2(b0.z, b0.w));
                  if (!(F16 && !X3F)) {
                    if (p0.x > 0.f) bb |= 1u << j;
                    if (p0.y > 0.f) bb |= 2u << j;
                    if (p1.x > 0.f) bb |= 4u << j;
                    if (p1.y > 0.f) bb |= 8u << j;
                  }
                  if (X3F) {
                    uint32_t a0, a1;
                    pack_hilo_h2(fmaxf(p0.x, 0.f), fmaxf(p0.y, 0.f), a0, vlo[j >> 1]);
                    pack_hilo_h2(fmaxf(p1.x, 0.f), fmaxf(p1.y, 0.f), a1, vlo[(j >> 1) + 1]);
                    v[j >> 1] = a0;
                    v[(j >> 1) + 1] = a1;
                  } else if (F16) {
                    // pairs go to v[0:16] (slots j/2, j/2+1 <= j were consumed already)
                    const uint32_t a0 = pack_relu_h2(p0.x, p0.y), a1 = pack_relu_h2(p1.x, p1.y);
                    {
                      bb |= pos_mask_h2(a0) & (0x00010001u << (j >> 1));
                      bb |= pos_mask_h2(a1) & (0x00010001u << ((j >> 1) + 1));
                    }
                    v[j >> 1] = a0;
                    v[(j >> 1) + 1] = a1;
                  } else {
                    v[j] = relu_tf32(p0.x); v[j + 1] = relu_tf32(p0.y); v[j + 2] = relu_tf32(p1.x); v[j + 3] = relu_tf32(p1.y);
                  }
                }
                bits[hh] = bb;
                if (F16)
                  tmem_st16(colX + half * 32 + 16 * hh, reinterpret_cast<uint32_t(&)[16]>(v));
                else
                  tmem_st32(colY + col0 + 32 * hh, v);
                if (X3F) tmem_st16(colX + 64 + half * 32 + 16 * hh, reinterpret_cast<uint32_t(&)[16]>(vlo));
              }
              if (GRAD && active) *reinterpret_cast<uint2*>(maskws + (it * 128 + row) * 4 + half * 2) = make_uint2(bits[0], bits[1]);
            }
            tmem_wait_st();
            tc_fence_before();
            ARR(); group_arrive(&a_ready[chain_id], lane);
            PH(3);
            // layer 3 epilogue: D3 (X[0:64]) + b3 -> the slots of this point that drew decoder k
            { STAT_T0(); acc_wait(&acc_ready[chain_id], ph_acc, lane); STAT_ADD(w_acc); }
            ph_acc ^= 1;
            tc_fence_after();
            PH(4); SKEW(18);
            if (wact) {
              uint32_t xv[32];
              tmem_ld32_sync((X3F ? colY : colX + (F16 ? 64 : 0)) + xc0, xv);
              float x[32];
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                const float4 bb = *reinterpret_cast<const float4*>(sw + OFF_B3 + xc0 + j);
                x[j] = __uint_as_float(xv[j]) + bb.x;
                x[j + 1] = __uint_as_float(xv[j + 1]) + bb.y;
                x[j + 2] = __uint_as_float(xv[j + 2]) + bb.z;
                x[j + 3] = __uint_as_float(xv[j + 3]) + bb.w;
              }
              // the slots of this point that drew decoder k (one compare for all four).  Even slot 2m: this point is the left
              // end of its segment (-> x1 row of the segment); odd slot 2m+1: right end of the previous one (-> x2 row)
              const uint32_t eq = active ? slot_match(sel, pt, k) : 0u;
#pragma unroll
              for (int j = 0; j < 2 * TC_MAX_M; ++j)
                if (eq & (1u << (8 * j))) {
                  float4* d = reinterpret_cast<float4*>(((j & 1) ? X2 + ((j >> 1) * W + pt - 1) * XD_STRIDE
                                                                 : X1 + ((j >> 1) * W + pt) * XD_STRIDE) + xc0);
#pragma unroll
                  for (int q = 0; q < 8; ++q)
                    if (q < nq) d[q] = make_float4(x[4 * q], x[4 * q + 1], x[4 * q + 2], x[4 * q + 3]);
                }
            }
            PH(5);
          }
          named_bar(3, EPI_THREADS);
          PH(7);

          // ============ x2 - x1, the energy, and the dE/dx operand tiles of the backward items ============
          if (GRAD) {
            // (1) The valid rows of one MC sample are contiguous in both buffers: a flat, fully coalesced pass over
            // 16-byte pieces (x2 from the workspace, x1 from shared memory or the workspace, the difference back in
            // place of x1), four independent pieces per thread in flight.  The energy is the plain sum of squares,
            // in a fixed order (deterministic).
            const int n4 = nseg * (XD_STRIDE / 4);
            if (!xl2) {
              // one curve, x1 in shared memory: both MC samples in one index space, eight x2 pieces (L2) in flight per thread
              constexpr int NV = XD_STRIDE / 4, NB = 8;
              const int ntot = Mb * n4;
              const float4* x2 = reinterpret_cast<const float4*>(X2);
              float4* x1 = reinterpret_cast<float4*>(X1);
              float e = 0.f;
              for (int i0 = t512; i0 < ntot; i0 += NB * EPI_THREADS) {
                float4 v[NB];
                int ad[NB];
#pragma unroll
                for (int j = 0; j < NB; ++j) {
                  const int idx = i0 + j * EPI_THREADS;
                  const int m = idx / n4;
                  ad[j] = idx < ntot ? m * W * NV + (idx - m * n4) : -1;
                  v[j] = ad[j] >= 0 ? __ldcg(x2 + ad[j]) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int j = 0; j < NB; ++j)
                  if (ad[j] >= 0) {
                    const float4 u = x1[ad[j]];
                    const float4 a = make_float4(v[j].x - u.x, v[j].y - u.y, v[j].z - u.z, v[j].w - u.w);
                    x1[ad[j]] = a;
                    e = fmaf(a.x, a.x, fmaf(a.y, a.y, fmaf(a.z, a.z, fmaf(a.w, a.w, e))));
                  }
              }
              PHW(20);
              e = warp_sum(e);
              if (lane == 0) s.red[320 + ew] = e;
              PHW(21);
            } else
            for (int jc = 0; jc < Gcur; ++jc) {      // the segments of one curve are contiguous rows: its energy
              float e = 0.f;
              for (int m = 0; m < Mb; ++m) {
                const float4* x2 = reinterpret_cast<const float4*>(X2 + size_t(m * W + jc * Wp) * XD_STRIDE);
                float4* x1 = reinterpret_cast<float4*>(X1 + size_t(m * W + jc * Wp) * XD_STRIDE);
                for (int i0 = t512; i0 < n4; i0 += 4 * EPI_THREADS) {
                  float4 v[4], u[4];
#pragma unroll
                  for (int j = 0; j < 4; ++j) {
                    const int i = i0 + j * EPI_THREADS;
                    v[j] = i < n4 ? __ldcg(x2 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
                    if (xl2) u[j] = i < n4 ? __ldcg(x1 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
                  }
#pragma unroll
                  for (int j = 0; j < 4; ++j) {
                    const int i = i0 + j * EPI_THREADS;
                    if (i < n4) {
                      if (!xl2) u[j] = x1[i];
                      const float4 a = make_float4(v[j].x - u[j].x, v[j].y - u[j].y, v[j].z - u[j].z, v[j].w - u[j].w);
                      x1[i] = a;
                      e = fmaf(a.x, a.x, fmaf(a.y, a.y, fmaf(a.z, a.z, fmaf(a.w, a.w, e))));
                    }
                  }
                }
              }
              e = warp_sum(e);
              if (lane == 0) s.red[320 + jc * 32 + ew] = e;
            }
            named_bar(3, EPI_THREADS);  // the differences are read by other threads below
            if (xl2) PHW(20);
            // (2) [only when the differences live in the workspace, xl2: from shared memory the backward items build
            // their dE/dx rows themselves -- inside an item the other chain hides the latency, a CTA-wide pass cannot;
            // measured 411 k vs 349 k spline-steps/s on the headline shape.]  One task = (item, row, 8 output columns): G = (2/M) * [sum over the segments whose RIGHT end is this
            // (point, decoder) of (x2 - x1)  -  sum over those whose LEFT end it is], written as one 16-byte piece of
            // the item's K-major operand tile in the workspace (fp16; 3-term mode: hi and lo tiles; tf32: two 16-byte
            // pieces of fp32).  The producer brings a tile into shared memory with bulk copies and B3 runs with its A
            // operand from shared memory: no per-item dE/dx build, no epilogue round trip in front of B3.
            const int ntask = xl2 ? nitems * 1024 : 0;
            const float gsc = F16 ? coefm * F16_GRAD_SCALE : coefm;
            // Eight consecutive threads = the eight 32-byte chunks of ONE row: a warp gathers four whole rows (a few
            // 128-byte lines) instead of one sector from each of 32 rows.  The gathers come from L2 -- or HBM: with
            // several curves per window the per-CTA buffers of a full grid exceed L2 -- so TB tasks per thread are in
            // flight: first the row lookups and the loads of each task's first matching slot (almost always the only
            // one), then the arithmetic; further slots of a task are fetched one after the other (rare).  Same order
            // of additions as the in-item build: slot order (sample 0: right end, left end; sample 1: right end, left end).
            constexpr int TB = VLG_TC_TILE_TB;
            for (int tb = t512; tb < ntask; tb += TB * EPI_THREADS) {
              float4 f0[TB], f1[TB];
              int ptv[TB];
              uint32_t mkv[TB];
#pragma unroll
              for (int u = 0; u < TB; ++u) {
                const int t0 = tb + u * EPI_THREADS;
                ptv[u] = -1;
                mkv[u] = 0u;
                f0[u] = f1[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (t0 < ntask) {
                  const int it = t0 >> 10, r = (t0 >> 3) & 127, c = t0 & 7;
                  const int k = ctl->item[it] & 0xFF, q0 = (ctl->item[it] >> 8) * 128;
                  const uint32_t cr = crow[k];
                  if (q0 + r < int(cr >> 16)) {
                    const int pt = rows[(cr & 0xFFFFu) + q0 + r];
                    ptv[u] = pt;
                    if (c < 7) {   // chunk 7 = zero padding (columns 56..63)
                      const uint32_t eq4 = slot_match(sel, pt, k);
                      // bit j: slot j in the order right end of segment pt-1 (sample 0), left end of segment pt (sample 0), ...
                      const uint32_t mk = ((eq4 >> 8) & 1u) | ((eq4 << 1) & 2u) | ((eq4 >> 22) & 4u) | ((eq4 >> 13) & 8u);
                      mkv[u] = mk;
                      if (mk) {
                        const int jj = __ffs(int(mk)) - 1;
                        const float4* src = reinterpret_cast<const float4*>(X1 + ptrdiff_t((jj >> 1) * W + pt - 1 + (jj & 1)) * XD_STRIDE + 8 * c);
                        f0[u] = xl2 ? __ldcg(src) : *src;
                        if (c < 6) f1[u] = xl2 ? __ldcg(src + 1) : *(src + 1);   // chunk 6 = columns 48..51 (+ zero padding up to 55)
                      }
                    }
                  }
                }
              }
#pragma unroll
              for (int u = 0; u < TB; ++u) {
                if (ptv[u] < 0) continue;
                const int t0 = tb + u * EPI_THREADS;
                const int it = t0 >> 10, r = (t0 >> 3) & 127, c = t0 & 7;
                const int pt = ptv[u];
                float g[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) g[q] = 0.f;
                uint32_t mk = mkv[u];
                float4 a0 = f0[u], a1 = f1[u];
                while (mk) {
                  const int jj = __ffs(int(mk)) - 1;
                  mk &= mk - 1u;
                  const float sg = (jj & 1) ? -1.f : 1.f;
                  g[0] = fmaf(sg, a0.x, g[0]); g[1] = fmaf(sg, a0.y, g[1]);
                  g[2] = fmaf(sg, a0.z, g[2]); g[3] = fmaf(sg, a0.w, g[3]);
                  g[4] = fmaf(sg, a1.x, g[4]); g[5] = fmaf(sg, a1.y, g[5]);
                  g[6] = fmaf(sg, a1.z, g[6]); g[7] = fmaf(sg, a1.w, g[7]);
                  if (mk) {   // a further slot of this row holds the same decoder
                    const int jn = __ffs(int(mk)) - 1;
                    const float4* src = reinterpret_cast<const float4*>(X1 + ptrdiff_t((jn >> 1) * W + pt - 1 + (jn & 1)) * XD_STRIDE + 8 * c);
                    a0 = xl2 ? __ldcg(src) : *src;
                    a1 = c < 6 ? (xl2 ? __ldcg(src + 1) : *(src + 1)) : make_float4(0.f, 0.f, 0.f, 0.f);
                  }
                }
#pragma unroll
                for (int q = 0; q < 8; ++q) g[q] *= gsc;
                unsigned char* tile = Gt + size_t(it) * GT_BYTES;
                if (F16) {
                  uint4 hi, lo;
                  if (X3B) {
                    pack_hilo_h2(g[0], g[1], hi.x, lo.x); pack_hilo_h2(g[2], g[3], hi.y, lo.y);
                    pack_hilo_h2(g[4], g[5], hi.z, lo.z); pack_hilo_h2(g[6], g[7], hi.w, lo.w);
                    *reinterpret_cast<uint4*>(tile + 16384 + (c * 128 + r) * 16) = lo;
                  } else {
                    hi = make_uint4(pack_h2(g[0], g[1]), pack_h2(g[2], g[3]), pack_h2(g[4], g[5]), pack_h2(g[6], g[7]));
                  }
                  *reinterpret_cast<uint4*>(tile + (c * 128 + r) * 16) = hi;
                } else {
                  uint4 v0, v1;
                  v0 = make_uint4(tf32_round_bits(__float_as_uint(g[0])), tf32_round_bits(__float_as_uint(g[1])),
                                  tf32_round_bits(__float_as_uint(g[2])), tf32_round_bits(__float_as_uint(g[3])));
                  v1 = make_uint4(tf32_round_bits(__float_as_uint(g[4])), tf32_round_bits(__float_as_uint(g[5])),
                                  tf32_round_bits(__float_as_uint(g[6])), tf32_round_bits(__float_as_uint(g[7])));
                  *reinterpret_cast<uint4*>(tile + ((2 * c) * 128 + r) * 16) = v0;
                  *reinterpret_cast<uint4*>(tile + ((2 * c + 1) * 128 + r) * 16) = v1;
                }
              }
            }
            if (xl2) fence_proxy_async_all();   // the tiles are read by the TMA engine (async proxy)
            if (xl2) PHW(21);
          } else {
            // forward-only kernel (also reports the polyline length, a sum of per-segment norms): 16 lanes
            // per (m, segment) entry, one 16-byte piece each; six entries per lane in flight.
            const int sub = lane & 15;
            constexpr int NV = XD_STRIDE / 4;   // 13 float4 per row
            constexpr int UNR = 6;
            const int nent = Mb * Wp;           // (m, local point) entries of one curve
            for (int jc = 0; jc < Gcur; ++jc) {
              float e = 0.f, l = 0.f;
              for (int base = ew * 2 + (lane >> 4); base < nent; base += 32 * UNR) {
                float4 v[UNR];
#pragma unroll
                for (int j = 0; j < UNR; ++j) {
                  const int ent = base + 32 * j;
                  const bool ok = ent < nent && (ent % Wp) < nseg && sub < NV;
                  const size_t r_ = size_t((ent / Wp) * W + jc * Wp + (ent % Wp)) * XD_STRIDE;
                  v[j] = ok ? __ldcg(reinterpret_cast<const float4*>(X2 + r_) + sub) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int j = 0; j < UNR; ++j) {
                  const int ent = base + 32 * j;
                  const bool ok = ent < nent && (ent % Wp) < nseg && sub < NV;
                  float q = 0.f;
                  if (ok) {
                    const size_t r_ = size_t((ent / Wp) * W + jc * Wp + (ent % Wp)) * XD_STRIDE;
                    const float4* up = reinterpret_cast<const float4*>(X1 + r_) + sub;
                    const float4 u = xl2 ? __ldcg(up) : *up;
                    const float4 a = make_float4(v[j].x - u.x, v[j].y - u.y, v[j].z - u.z, v[j].w - u.w);
                    q = fmaf(a.x, a.x, fmaf(a.y, a.y, fmaf(a.z, a.z, a.w * a.w)));
                  }
#pragma unroll
                  for (int o = 8; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
                  if (sub == 0) { e += q; l += sqrtf(q); }
                }
              }
              e = warp_sum(e);
              l = warp_sum(l);
              if (lane == 0) { s.red[320 + jc * 32 + ew] = e; s.red[320 + jc * 32 + 16 + ew] = l; }
            }
          }
          if (GRAD) {
            named_bar(3, EPI_THREADS);            // every tile of the window is written (and fenced for the async proxy)
            if (xl2 && t512 == 0) mbar_arrive(g_ready);  // -> the producers may bring them into shared memory
          }
          PH(8);

          if (GRAD) {
            // =============================== backward ===============================
            // dz of a (point, decoder) row = sum of its two half-threads' partials; it goes to the cell of the FIRST draw
            // slot of the point that holds this decoder -- each cell is written exactly once, and the <= 4 cells of a
            // point are added in slot order afterwards: the result does not depend on which item / chain / window-mate
            // a row was processed with.  The halves meet through dzx one item later (the chain's next MMA round trip
            // is a barrier between the group's threads).
            // G = dE/dx_k of a row, columns xc0 .. xc0+31, packed for B3 and stored to tensor memory.  Single-term fp16
            // backward (G_AHEAD): G lives in X[64:96], which no other backward operand or accumulator touches, so the
            // NEXT item's rows are built and stored while B2 of the current item runs -- no registers are held across the
            // epilogue phases (the 3-term format needs X[64:128] for residual operands and builds G in place, X[0:32]).
            constexpr bool G_AHEAD = F16 && !X3B && !xl2 && VLG_TC_G_AHEAD;
            const uint32_t gcolX = colX + (G_AHEAD ? 64u : 0u);
            auto build_g = [&](int k, int pt, bool active, bool wact) {
                if (wact) {
                  float g[32];
  #pragma unroll
                  for (int j = 0; j < 32; ++j) g[j] = 0.f;
                  const uint32_t eq = active ? slot_match(sel, pt, k) : 0u;
#pragma unroll
                  for (int m = 0; m < TC_MAX_M; ++m) {     // same order of additions as ever: right end, then left end, per sample
                    if (eq & (0x100u << (16 * m))) {
                      const float4* d = reinterpret_cast<const float4*>(X1 + (m * W + pt - 1) * XD_STRIDE + xc0);
  #pragma unroll
                      for (int q = 0; q < 8; ++q)
                        if (q < nq) {
                          const float4 v = d[q];
                          g[4 * q] += v.x; g[4 * q + 1] += v.y; g[4 * q + 2] += v.z; g[4 * q + 3] += v.w;
                        }
                    }
                    if (eq & (0x1u << (16 * m))) {
                      const float4* d = reinterpret_cast<const float4*>(X1 + (m * W + pt) * XD_STRIDE + xc0);
  #pragma unroll
                      for (int q = 0; q < 8; ++q)
                        if (q < nq) {
                          const float4 v = d[q];
                          g[4 * q] -= v.x; g[4 * q + 1] -= v.y; g[4 * q + 2] -= v.z; g[4 * q + 3] -= v.w;
                        }
                    }
                  }
                  if (F16) {
                    uint32_t v[16], vl[X3B ? 16 : 1];
  #pragma unroll
                    for (int j = 0; j < 16; ++j) {
                      const float g0 = (coefm * F16_GRAD_SCALE) * g[2 * j], g1 = (coefm * F16_GRAD_SCALE) * g[2 * j + 1];
                      if (X3B)
                        pack_hilo_h2(g0, g1, v[j], vl[j]);
                      else
                        v[j] = pack_h2(g0, g1);
                    }
                    tmem_st16(gcolX + half * 16, v);
                    if (X3B) tmem_st16(colX + 64 + half * 16, reinterpret_cast<uint32_t(&)[16]>(vl));
                  } else {
                    uint32_t v[32];
  #pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = tf32_round_bits(__float_as_uint(coefm * g[j]));
                    tmem_st32(colX + xc0, v);
                  }
                }
            };
            int pend_pt = -1, pend_slot = 0;
            // row of this thread in item `it2` (decoder, point, flags) -- for the look-ahead build
            auto item_row = [&](int it2, int& k2, int& pt2, bool& act2, bool& wact2) {
              k2 = ctl->item[it2] & 0xFF;
              const int q02 = (ctl->item[it2] >> 8) * 128;
              const uint32_t cr2 = crow[k2];
              act2 = q02 + row < int(cr2 >> 16);
              wact2 = q02 + (warp & 3) * 32 < int(cr2 >> 16);
              pt2 = act2 ? rows[(cr2 & 0xFFFFu) + q02 + row] : 0;
            };
            if (G_AHEAD && chain_id < nitems) {   // the first item of the chain
              int k2, pt2; bool a2, w2;
              item_row(chain_id, k2, pt2, a2, w2);
              build_g(k2, pt2, a2, w2);
              tmem_wait_st();
              tc_fence_before();
              ARR(); group_arrive(&a_ready[chain_id], lane);
            }
            for (int it = chain_id; it < nitems; it += 2) {
              const int k = ctl->item[it] & 0xFF, q0 = (ctl->item[it] >> 8) * 128;
              const uint32_t cr = crow[k];
              const bool active = q0 + row < int(cr >> 16);
              const bool wact = q0 + (warp & 3) * 32 < int(cr >> 16);
              const int pt = active ? rows[(cr & 0xFFFFu) + q0 + row] : 0;
              mbar_wait(&sw_full[chain_id * SW_SLOTS + (swj % SW_SLOTS)], (swj / SW_SLOTS) & 1u);
              if (!F16) named_bar(bar_id, GROUP_THREADS);
              const float* sw = swbuf + (swj % SW_SLOTS) * 576;
              ++swj;
              const float2 z = s.zs[pt];
              const float2 zx2 = make_float2(z.x, z.x), zy2 = make_float2(z.y, z.y);
              // mask words for E-B3 (the L2 round trip overlaps the first MMA)
              uint2 bits = make_uint2(0u, 0u);
              if (active) bits = *reinterpret_cast<const uint2*>(maskws + (it * 128 + row) * 4 + half * 2);
              if (xl2) {
                // B3 takes its A operand (the dE/dx tile) from shared memory: nothing to build here.  This arrive
                // only tells the issuer that the chain's accumulator columns are free (all tcgen05.ld of the
                // previous item are complete in program order).
                tc_fence_before();
                ARR(); group_arrive(&a_ready[chain_id], lane);
              } else {
                // G = dE/dx_k (this point), columns xc0 .. xc0+31 -> tensor memory (see build_g)
                if (!G_AHEAD) {
                  build_g(k, pt, active, wact);
                  tmem_wait_st();
                  tc_fence_before();
                  ARR(); group_arrive(&a_ready[chain_id], lane);
                }
              }
              PH(9);
              // dh2 = (G W3) * mask2 -> A4 (Y, in place)
              { STAT_T0(); acc_wait(&acc_ready[chain_id], ph_acc, lane); STAT_ADD(w_acc); }
              ph_acc ^= 1;
              tc_fence_after();
              PH(10); SKEW(19);
              if (half == 0 && pend_pt >= 0) {   // the previous item's row: both halves are in dzx now
                const float2 u0 = s.dzx[(chain_id * 2 + 0) * 128 + row], u1 = s.dzx[(chain_id * 2 + 1) * 128 + row];
                s.dzs[pend_slot * W + pend_pt] = make_float2(u0.x + u1.x, u0.y + u1.y);
              }
              if (wact) {
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                  uint32_t v[32];
                  tmem_ld32_sync(colY + col0 + 32 * hh, v);
                  const uint32_t mb = hh ? bits.y : bits.x;
                  if (F16) {
                    uint32_t vl[X3B ? 16 : 1];
#pragma unroll
                    for (int j = 0; j < 32; j += 2) {
                      if (!X3F) {
                        // bits p, 16+p -> 0xFFFF lane masks (no carries: 1 * 0xFFFF, 0x10000 * 0xFFFF)
                        const uint32_t lanes = ((mb >> (j >> 1)) & 0x00010001u) * 0xFFFFu;
                        v[j >> 1] = pack_h2(__uint_as_float(v[j]), __uint_as_float(v[j + 1])) & lanes;
                        continue;
                      }
                      const float a0 = ((mb >> j) & 1u) ? __uint_as_float(v[j]) : 0.f;
                      const float a1 = ((mb >> (j + 1)) & 1u) ? __uint_as_float(v[j + 1]) : 0.f;
                      if (X3B)
                        pack_hilo_h2(a0, a1, v[j >> 1], vl[j >> 1]);
                      else
                        v[j >> 1] = pack_h2(a0, a1);   // j/2 <= j: slot already consumed
                    }
                    tmem_st16(colX + half * 32 + 16 * hh, reinterpret_cast<uint32_t(&)[16]>(v));
                    if (X3B) tmem_st16(colX + 64 + half * 32 + 16 * hh, reinterpret_cast<uint32_t(&)[16]>(vl));
                  } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = ((mb >> j) & 1u) ? tf32_round_bits(v[j]) : 0u;
                    tmem_st32(colY + col0 + 32 * hh, v);
                  }
                }
              }
              tmem_wait_st();
              tc_fence_before();
              ARR(); group_arrive(&a_ready[chain_id], lane);
              PH(11);
              if (G_AHEAD && it + 2 < nitems) {   // under B2 of this item: the next item's dE/dx rows -> X[64:96]
                int k2, pt2; bool a2, w2;
                item_row(it + 2, k2, pt2, a2, w2);
                build_g(k2, pt2, a2, w2);
                tmem_wait_st();
              }
              // dh1 = (dh2 W2) * mask1 (recomputed); dz[point] += dh1 W1 over this thread's 64 hidden units
              { STAT_T0(); acc_wait(&acc_ready[chain_id], ph_acc, lane); STAT_ADD(w_acc); }
              ph_acc ^= 1;
              tc_fence_after();
              PH(12); SKEW(20);
              if (wact) {
                float2 ax = make_float2(0.f, 0.f), ay = make_float2(0.f, 0.f);
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                  uint32_t v[32];
                  tmem_ld32_sync((F16 ? colY : colX) + col0 + 32 * hh, v);
#pragma unroll
                  for (int j = 0; j < 32; j += 4) {   // 16-byte loads of the (warp-uniform) layer-1 weights
                    const int c = col0 + 32 * hh + j;
                    const float4 wx4 = *reinterpret_cast<const float4*>(sw + OFF_W1X + c);
                    const float4 wy4 = *reinterpret_cast<const float4*>(sw + OFF_W1Y + c);
                    const float4 bb4 = *reinterpret_cast<const float4*>(sw + OFF_B1 + c);
#pragma unroll
                    for (int e = 0; e < 2; ++e) {     // same pair order as ever: (c, c+1), then (c+2, c+3)
                      const float2 wx = e ? make_float2(wx4.z, wx4.w) : make_float2(wx4.x, wx4.y);
                      const float2 wy = e ? make_float2(wy4.z, wy4.w) : make_float2(wy4.x, wy4.y);
                      const float2 bb = e ? make_float2(bb4.z, bb4.w) : make_float2(bb4.x, bb4.y);
                      const float2 h = __ffma2_rn(wy, zy2, __ffma2_rn(wx, zx2, bb));
                      const float2 dh = make_float2(h.x > 0.f ? __uint_as_float(v[j + 2 * e]) : 0.f,
                                                    h.y > 0.f ? __uint_as_float(v[j + 2 * e + 1]) : 0.f);
                      ax = __ffma2_rn(dh, wx, ax);
                      ay = __ffma2_rn(dh, wy, ay);
                    }
                  }
                }
                if (active) {
                  constexpr float unscale = F16 ? 1.f / F16_GRAD_SCALE : 1.f;
                  s.dzx[(chain_id * 2 + half) * 128 + row] = make_float2((ax.x + ax.y) * unscale, (ay.x + ay.y) * unscale);
                }
              }
              pend_pt = -1;
              if (active && half == 0) {
                pend_pt = pt;
                pend_slot = (__ffs(int(slot_match(sel, pt, k))) - 1) >> 3;   // first draw slot of the point that holds decoder k
              }
              PH(13);
              if (G_AHEAD && it + 2 < nitems) {   // D5 is in registers (tcgen05.wait::ld): B3 of the next item may overwrite Y
                tc_fence_before();
                ARR(); group_arrive(&a_ready[chain_id], lane);
              }
            }
            named_bar(3, EPI_THREADS);
            PH(14);
            if (half == 0 && pend_pt >= 0) {     // the last item of each chain
              const float2 u0 = s.dzx[(chain_id * 2 + 0) * 128 + row], u1 = s.dzx[(chain_id * 2 + 1) * 128 + row];
              s.dzs[pend_slot * W + pend_pt] = make_float2(u0.x + u1.x, u0.y + u1.y);
            }
          }
          named_bar(3, EPI_THREADS);
          if (t512 == 0) mbar_arrive(&ctl_free[buf]);   // done with this window's draws and lists: the buffer may be rewritten
          PHW(22);
          // ---- energy of the window per curve; d(omega) += P^T dz over the points of the window ----
          if (t512 < Gcur) {
            float ee = 0.f, ll = 0.f;
            for (int w = 0; w < 16; ++w) { ee += s.red[320 + t512 * 32 + w]; ll += s.red[320 + t512 * 32 + 16 + w]; }
            s.etot[2 * t512] += ee;
            if (!GRAD) s.etot[2 * t512 + 1] += ll;
          }
          if (GRAD) {
            // chunks of 512 points, one point per thread; a warp's 32 points belong to one curve (Wp % 32 == 0
            // whenever a window holds several curves); per chunk the 16 warp partials are added to their curves'
            // gradients in warp order by one thread per coefficient (fixed order)
            const int wpos = t512 >> 5;
            for (int ch = 0; ch < nchunk; ++ch) {
              const int pt = ch * 512 + t512;
              float P[MAX_KB];
              float dx = 0.f, dy = 0.f;
              if (pt < W) {
                const int i = pt - (pt / Wp) * Wp;
                design_row(p.t[min(seg0 + i, T - 1)], n_poly, Kb, s.basis, P);
                const float2 d0 = s.dzs[pt], d1 = s.dzs[W + pt], d2 = s.dzs[2 * W + pt], d3 = s.dzs[3 * W + pt];
                dx = (d0.x + d1.x) + (d2.x + d3.x);
                dy = (d0.y + d1.y) + (d2.y + d3.y);
              } else {
#pragma unroll
                for (int k = 0; k < MAX_KB; ++k) P[k] = 0.f;
              }
#pragma unroll
              for (int k = 0; k < MAX_KB; ++k)
                if (k < Kb) {
                  const float cx = warp_sum(P[k] * dx), cy = warp_sum(P[k] * dy);
                  if (lane == 0) { s.red[wpos * 20 + 2 * k] = cx; s.red[wpos * 20 + 2 * k + 1] = cy; }
                }
              named_bar(3, EPI_THREADS);
              PHW(23);
              if (t512 < 2 * Kb) {
                for (int w = 0; w < 16; ++w) {
                  const int p0 = ch * 512 + w * 32;
                  if (p0 < W) s.gacc[(p0 / Wp) * 20 + t512] += s.red[w * 20 + t512];
                }
              }
              named_bar(3, EPI_THREADS);
            }
            // gradient-output mode: dE/da += sum (1-t) dz, dE/db += sum t dz -- the design row extended by (1-t, t),
            // in a second pass of the same shape
            if (GOUT) {
              for (int ch = 0; ch < nchunk; ++ch) {
                const int pt = ch * 512 + t512;
                float dx = 0.f, dy = 0.f, tp = 0.f;
                if (pt < W) {
                  tp = p.t[min(seg0 + pt - (pt / Wp) * Wp, T - 1)];
                  const float2 d0 = s.dzs[pt], d1 = s.dzs[W + pt], d2 = s.dzs[2 * W + pt], d3 = s.dzs[3 * W + pt];
                  dx = (d0.x + d1.x) + (d2.x + d3.x);
                  dy = (d0.y + d1.y) + (d2.y + d3.y);
                }
                const float ax = warp_sum((1.0f - tp) * dx), ay = warp_sum((1.0f - tp) * dy);
                const float bx = warp_sum(tp * dx), by = warp_sum(tp * dy);
                float* r = s.red + wpos * 20;
                if (lane == 0) { r[0] = ax; r[1] = ay; r[2] = bx; r[3] = by; }
                named_bar(3, EPI_THREADS);
                if (t512 < 4) {
                  for (int w = 0; w < 16; ++w) {
                    const int p0 = ch * 512 + w * 32;
                    if (p0 < W) s.om[(p0 / Wp) * OM_STRIDE + 2 * MAX_KB + t512] += s.red[w * 20 + t512];
                  }
                }
                named_bar(3, EPI_THREADS);
              }
            }
          } else {
            named_bar(3, EPI_THREADS);
          }
          PH(15);
        }  // windows

        if (t512 < Gcur) write_energy(p, n0 + t512, step, s.etot[2 * t512], s.etot[2 * t512 + 1], &queue[1]);
        if (GOUT) {
          const int ncol = 2 * Kb + 4;
          if (t512 < Gcur * ncol) {
            const int j = t512 / ncol, c = t512 - j * ncol;
            write_grad(p, n0 + j, c, c < 2 * Kb ? s.gacc[j * 20 + c] : s.om[j * OM_STRIDE + 2 * MAX_KB + c - 2 * Kb],
                       &queue[1]);
          }
        } else if (MODE == StepMode::Optimize && t512 < Gcur * 2 * Kb) {
          const int j = t512 / (2 * Kb), c = t512 - j * 2 * Kb;
          const float* ab = s.pab + 4 * j;
          penalty_adam_step(p, step, c, s.gacc[j * 20 + c], s.basis, s.coef + j * 64, make_float2(ab[0], ab[1]),
                            make_float2(ab[2], ab[3]), s.om + j * OM_STRIDE);
        }
        named_bar(3, EPI_THREADS);
      }  // steps

      if (MODE == StepMode::Optimize && t512 < Gcur * 2 * Kb) {
        const int j = t512 / (2 * Kb), c = t512 - j * 2 * Kb;
        write_back(p, n0 + j, c, s.om + j * OM_STRIDE, &queue[1]);
        __threadfence();
      }
      named_bar(3, EPI_THREADS);
      if (t512 == 0) {
        const unsigned int v = unsigned(chunk) + 1u;
        asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(&queue[64 + grp]), "r"(v) : "memory");
      }
    }  // work units
#ifdef VLG_TC_STATS
    if (tg == 0 && blockIdx.x < 1024) g_tc_stats[blockIdx.x * 8 + 4 + chain_id * 2] = w_acc;
#endif
    PH_FLUSH();
    (void)w_acc;
  } else {
    // ================= window setup: draws, row lists and item lists, one window ahead of the epilogue =================
    // Runs through the same (work unit, step, window, sample block) sequence as the epilogue.  Nothing here depends on
    // a window's results: the draws are counter-based (or read from p.draws), the lists depend on the draws only.
    // Window w is built into buffer w & 1 once every consumer -- producers, issuer, epilogue -- is done with window
    // w - 2 (ctl_free), and announced on win_ready[w & 1].
    long wseq = 0;                              // windows set up so far
    bool bad_draw = false;                      // an explicit draw was >= K (clamped)
    unsigned long long n_items = 0, n_rows = 0; // 128-row items / occupied rows (launch statistics)
    const int selw = tc_sel_words(W);
#ifdef VLG_TC_STATS
    long long t_busy = 0, t_free = 0;
#endif
    auto claim_buffer = [&]() {
#ifdef VLG_TC_STATS
      const long long t0 = clock64();
#endif
      if (wseq >= 2) mbar_wait(&ctl_free[wseq & 1], uint32_t(((wseq >> 1) - 1) & 1));
#ifdef VLG_TC_STATS
      t_free += clock64() - t0;
#endif
    };
    unsigned int unit;
    for (;;) {
      claim_buffer();
      unit = 0;
      if (lane == 0) unit = atomicAdd(&queue[0], 1u);
      unit = __shfl_sync(0xffffffffu, unit, 0);
      if (unit >= total_units) break;
      const int grp = int(unit % ngroups);
      const int n0 = grp * G, Gcur = XL2 ? min(G, p.N - n0) : 1;
      const int chunk = int(unit / ngroups);
      const int step_lo = chunk * unit_steps, step_hi = min(p.steps, step_lo + unit_steps);
      // one weight set per window: per-curve sets (decoder_base) are only launched with G = 1
      const int dec_base = curve_dec_base(p, n0, lane == 0, &queue[1]);
      for (int step = step_lo; step < step_hi; ++step)
        for (int win = 0; win < nwin; ++win)
          for (int mb = 0; 2 * mb < Mtot; ++mb, ++wseq) {
            const int Mb = min(TC_MAX_M, Mtot - 2 * mb);   // samples of this block
            const int seg0 = win * WSEG;
            const int nseg = min(WSEG, T - 1 - seg0);     // segments of every curve in this window
            const int buf = int(wseq & 1);
            claim_buffer();
#ifdef VLG_TC_STATS
            const long long t0 = clock64();
#endif
            uint8_t* sel = s.sel + size_t(buf) * selw * 4;
            uint16_t* rows = s.rows + size_t(buf) * 2 * M * W;
            uint32_t* crow = s.crow + buf * TC_MAX_K;
            WinCtl* ctl = &s.ctl[buf];
            // ---- draws: one word per point (lane = point).  Words W .. selw-1 hold no draw (255) ----
            for (int i = W + lane; i < selw; i += 32) reinterpret_cast<uint32_t*>(sel)[i] = 0xFFFFFFFFu;
            __syncwarp();
            for (int pt = lane; pt < W; pt += 32) {
              const int j = pt / Wp, i = pt - j * Wp;   // point pt = curve j = pt / Wp, local index i
              const bool seg_ok = i < nseg && j < Gcur;
              const int n = n0 + j;
              if (p.draws != nullptr) {
                for (int m = 0; m < Mb; ++m)
                  for (int role = 0; role < 2; ++role) {
                    sel[4 * (pt + role) + 2 * m + role] = seg_ok ? explicit_draw(p.draws, p.steps, Mtot, T, K, n, step, 2 * mb + m, role, seg0 + i, bad_draw) : 255;
                  }
                if (Mb < 2) { sel[4 * pt + 2] = 255; sel[4 * pt + 7] = 255; }
              } else {
                uint32_t d[4] = {255u, 255u, 255u, 255u};
                if (seg_ok)
                  counter_draws4(p.seed, uint32_t(p.curve_id0 + n), uint32_t(p.step0 + step), uint32_t(seg0 + i), uint32_t(mb),
                                 uint32_t(K), d);
                for (int q = 0; q < 4; ++q) sel[4 * (pt + (q & 1)) + q] = (q >> 1) < Mb ? uint8_t(d[q]) : uint8_t(255);
              }
              if (pt == 0) { sel[1] = 255; sel[3] = 255; }   // no segment ends at the first point
            }
            __syncwarp();
            // ---- per-decoder row lists, in increasing point order ----
            // Item membership must not depend on thread timing: a decoder drawn by more than 128 points of the
            // window is split into several items, which run on different chains, and the chains' dz partial sums
            // are added in a fixed order -- so WHICH points share an item fixes the fp32 summation grouping.
            // Lane = decoder (32 at a time): a count pass over the points, scans over the lanes for the list
            // offsets and item numbers, then a pass that appends every matching point to the lane's own list.
            // A point enters a decoder's list once, whichever of its draw slots hold the decoder.
            const uint4* sel4 = reinterpret_cast<const uint4*>(sel);
            auto holds = [](uint32_t w, uint32_t kp) {   // some byte of w equals the byte of kp (exact zero-byte test)
              const uint32_t y = w ^ kp;
              return ((y - 0x01010101u) & ~y & 0x80808080u) != 0u;
            };
            int off_carry = 0, ni_carry = 0;
            for (int k0 = 0; k0 < K; k0 += 32) {
              const int k = k0 + lane;   // k >= K matches no byte: draws are < K or 255
              const uint32_t kp = uint32_t(k) * 0x01010101u;
              int cnt = 0;
              for (int q = 0; 4 * q < W; ++q) {
                const uint4 v = sel4[q];
                cnt += int(holds(v.x, kp)) + int(holds(v.y, kp)) + int(holds(v.z, kp)) + int(holds(v.w, kp));
              }
              const int nit = (cnt + 127) >> 7;
              int so = cnt, si = nit;   // inclusive scans over the lanes
#pragma unroll
              for (int o = 1; o < 32; o <<= 1) {
                const int a = __shfl_up_sync(0xffffffffu, so, o), b = __shfl_up_sync(0xffffffffu, si, o);
                if (lane >= o) { so += a; si += b; }
              }
              const int roff = off_carry + so - cnt;
              if (k < K) {
                crow[k] = uint32_t(roff) | (uint32_t(cnt) << 16);
                const int i0 = ni_carry + si - nit;
                for (int q = 0; q < nit; ++q) ctl->item[i0 + q] = uint16_t(k | (q << 8));
              }
              off_carry += __shfl_sync(0xffffffffu, so, 31);
              ni_carry += __shfl_sync(0xffffffffu, si, 31);
              uint16_t* out = rows + roff;
              for (int q = 0; 4 * q < W; ++q) {
                const uint4 v = sel4[q];
                if (holds(v.x, kp)) *out++ = uint16_t(4 * q);
                if (holds(v.y, kp)) *out++ = uint16_t(4 * q + 1);
                if (holds(v.z, kp)) *out++ = uint16_t(4 * q + 2);
                if (holds(v.w, kp)) *out++ = uint16_t(4 * q + 3);
              }
            }
            if (lane == 0) {
              ctl->nitems = ni_carry;
              ctl->base = dec_base;
              ctl->unit = unit;
              n_items += unsigned(ni_carry);
              n_rows += unsigned(off_carry);
            }
            __threadfence_block();
            __syncwarp();
            if (lane == 0) mbar_arrive(&win_ready[buf]);
#ifdef VLG_TC_STATS
            t_busy += clock64() - t0;
#endif
          }
    }
    // no more work: an item list with no items, in the buffer of the next window
    if (lane == 0) {
      s.ctl[wseq & 1].nitems = -1;
      s.ctl[wseq & 1].unit = unit;
      __threadfence_block();
      mbar_arrive(&win_ready[wseq & 1]);
    }
    if (bad_draw) atomicOr(&queue[1], unsigned(VLG_STATUS_BAD_DRAW));
    if (lane == 0) {   // launch statistics for vlg_workspace_counters (words [2..5] of the header)
      atomicAdd(reinterpret_cast<unsigned long long*>(queue + 2), n_items);
      atomicAdd(reinterpret_cast<unsigned long long*>(queue + 4), n_rows);
    }
#ifdef VLG_TC_STATS
    if (lane == 0 && blockIdx.x < 1024) {
      g_tc_stats[blockIdx.x * 8 + 0] = t_busy;
      g_tc_stats[blockIdx.x * 8 + 1] = t_free;
    }
#endif
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem, 512);
}

// Launch plan.  Window length: as few 128-row items per curve as possible.  A decoder is drawn by a point with
// probability p = 1 - (1 - 1/K)^(2M); its row count n in a window of W points is ~Binomial(W, p) and it
// costs ceil(n/128) items.  Evaluate the expected item count for every admissible number of windows, for both
// homes of the left-end outputs / differences: shared memory (xl2 = 0; 208 M bytes per point limit the window)
// or the L2-resident workspace (xl2 = 1; any window up to TC_MAX_W points, but the dE/dx tile pass then sits on
// L2 latency: measured +45 % per item on the headline shape).
struct TcPlan {
  int W, nst, xl2, G;   // W = points per window (all curves), G = curves per window
};
static TcPlan tc_plan(int T, int K, int M, bool allow_multi) {
  if (M > TC_MAX_M) M = TC_MAX_M;   // samples per block
  const double p = 1.0 - pow(1.0 - 1.0 / K, 2.0 * M);
  const int segs = T - 1;
  int force_nwin = 0, force_xl2 = -1, force_g = 0;
  if (const char* env = getenv("VLG_TC_WINDOW")) force_nwin = atoi(env);   // tuning overrides
  if (const char* env = getenv("VLG_TC_XL2")) force_xl2 = atoi(env);
  if (const char* env = getenv("VLG_TC_G")) force_g = atoi(env);
  TcPlan best = {0, 0, 0, 1};
  double best_cost = 1e300;
  for (int xl2 = 0; xl2 < 2; ++xl2) {
    if (force_xl2 >= 0 && xl2 != force_xl2) continue;
    // one curve per window, nwin windows along the curve
    for (int nwin = 1; nwin <= segs; ++nwin) {
      const int w = (segs + nwin - 1) / nwin + 1;  // points per window
      if (force_nwin >= 1 && nwin != force_nwin) {
        if (w <= 128) break;
        continue;
      }
      if (w <= TC_MAX_W && force_g <= 1) {
        const int nst = tc_stages(w, K, M, xl2);
        if (nst >= 2) {
          double cost = nwin * (K * expected_items(w, p) + 0.35);  // + per-window fixed cost in item units
          if (nst == 2) cost *= 1.04;               // a two-stage weight ring cannot hold a whole GEMM's weights
          if (xl2) cost *= 1.45;
          if (cost < best_cost) { best_cost = cost; best = {w, nst, xl2, 1}; }
        }
      }
      if (w <= 128) break;
    }
    // G whole curves per window (short curves, many decoders: one curve alone leaves the 128-row items almost empty)
    if (xl2 && allow_multi && T % 32 == 0)
      for (int g = 2; g <= TC_MAX_G && g * T <= TC_MAX_WG; ++g) {
        if (force_g >= 2 && g != force_g) continue;
        const int w = g * T;
        const int nst = tc_stages(w, K, M, 1);
        if (nst < 2) continue;
        double cost = (K * expected_items(w, p) + 0.35) / g * 1.45;
        if (nst == 2) cost *= 1.04;
        if (cost < best_cost) { best_cost = cost; best = {w, nst, 1, g}; }
      }
  }
  return best;  // W == 0: does not fit
}

size_t tc_workspace_bytes(int N, int T, int K, int M) {
  if (K > TC_MAX_K) return 0;
  if (M > TC_MAX_M) M = TC_MAX_M;   // buffers are sized for one block of samples
  const TcPlan pl = tc_plan(T, K, M, true);   // the multi-curve plan needs at least as much as the single-curve one
  const TcPlan p1 = tc_plan(T, K, M, false);
  const size_t a = tc_ws_cta_words(K, M, pl.W), b = tc_ws_cta_words(K, M, p1.W);
  return tc_queue_words(N) * 4 + size_t(persistent_grid(N)) * (a > b ? a : b) * 4;
}

#ifdef VLG_TC_STATS
extern "C" int vlg_debug_tc_stats(long long* host_out, int n) {
  return cudaMemcpyFromSymbol(host_out, g_tc_stats, size_t(n) * 8 * sizeof(long long)) == cudaSuccess ? 0 : -3;
}
extern "C" int vlg_debug_tc_phase(long long* host_out, int n) {
  return cudaMemcpyFromSymbol(host_out, g_tc_phase, size_t(n) * 48 * sizeof(long long)) == cudaSuccess ? 0 : -3;
}
#endif

cudaError_t launch_tc(const StepParams& p, cudaStream_t stream) {
  if (p.precision < 1 || p.precision > 4) return cudaErrorNotSupported;
  const int fmt = p.precision == 1 ? FMT_TF32 : p.precision == 3 ? FMT_F16 : p.precision == 4 ? FMT_F16X3F : FMT_F16X3;
  if (p.K > TC_MAX_K || p.M < 1) return cudaErrorNotSupported;
  const int Mc = p.M > TC_MAX_M ? TC_MAX_M : p.M;
  const TcPlan pl = tc_plan(p.T, p.K, Mc, p.dec_base == nullptr);   // per-curve weight sets: one curve per window
  const int W = pl.W, nst = pl.nst, xl2 = pl.xl2, G = pl.G;
  if (W < 2 || nst < 2) return cudaErrorNotSupported;
  if (p.workspace == nullptr || p.workspace_bytes < tc_workspace_bytes(p.N, p.T, p.K, p.M)) return cudaErrorInvalidValue;
  const size_t smem = tc_smem_fixed_bytes(W, p.K, Mc, xl2) + size_t(2) * nst * STAGE_BYTES;
  const int ngroups = (p.N + G - 1) / G;
  const int grid = persistent_grid(ngroups);
  StepParams q = p;
  // chunks of a curve (group) per launch: at least 4, and enough work units (~48 per CTA) that the last wave's
  // tail -- at most one unit -- stays a small fraction of the launch
  int nchunks = (48 * grid + ngroups - 1) / ngroups;
  if (nchunks < 4) nchunks = 4;
  if (nchunks > q.steps) nchunks = q.steps;
  q.unit_steps = (q.steps + nchunks - 1) / nchunks;
  cudaError_t e = cudaMemsetAsync(p.workspace, 0, tc_queue_words(p.N) * 4, stream);
  if (e != cudaSuccess) return e;
  auto launch = [&](auto kernel) -> cudaError_t {
    cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (err != cudaSuccess) return err;
    kernel<<<grid, TC_THREADS, smem, stream>>>(q, nst, W, G);
    return cudaGetLastError();
  };
  auto by_fmt = [&](auto mode_c, auto xl2_c) -> cudaError_t {
    constexpr StepMode MODE = decltype(mode_c)::value;
    constexpr bool X = decltype(xl2_c)::value;
    if (fmt == FMT_TF32) return launch(tc_curve_kernel<MODE, FMT_TF32, X>);
    if (fmt == FMT_F16) return launch(tc_curve_kernel<MODE, FMT_F16, X>);
    if constexpr (MODE != StepMode::Energy) {   // forward only: the mixed format IS the 3-term format
      if (fmt == FMT_F16X3F) return launch(tc_curve_kernel<MODE, FMT_F16X3F, X>);
    }
    return launch(tc_curve_kernel<MODE, FMT_F16X3, X>);
  };
  return with_mode(p.mode, [&](auto mode_c) {
    return xl2 ? by_fmt(mode_c, std::true_type{}) : by_fmt(mode_c, std::false_type{});
  });
}

}  // namespace vlg
