// fp32 (CUDA-core FFMA) geodesic step kernel: the <=1e-4-per-step variant and the one
// the single-decoder path (BASELINE config 2) needs, since 11-bit tensor-core operands destroy
// the tiny adjacent-point differences there (SURVEY hard part 1).
//
// Persistent CTAs (one per SM), each walking curves n = blockIdx.x, +gridDim.x, ... over `steps`
// Adam steps.  Per step the curve is cut into windows of W points (W-1 segments; neighbouring
// windows share one point).  ROW COMPACTION as in the tensor-core kernel: per decoder only the points
// of the window that drew it (as left or right end of a segment) are gathered into the rows of
// 128-row "items"; a (point, decoder) pair nobody drew is never evaluated (the reference evaluates
// all K x T pairs and multiplies two thirds of them by zero).  Per window:
//   draws -> per-decoder row lists -> forward items (register-tiled 128x128x128 / 128x64x128
//   SGEMMs, activations staged transposed+swizzled in shared memory, weights streamed from L2 in
//   16-row slabs) -> selected outputs accumulate into Diff[m][segment] = x_{d2}(t+1) - x_{d1}(t)
//   -> energy (and poly-line length) -> backward items (input gradient only, layer-2 ReLU masks as
//   bits in an L2-resident workspace, layer-1 mask recomputed) -> dz per point -> d(omega).
// Then the end-point penalty gradient and Adam, all in shared memory; omega/m/v touch HBM
// once per launch.  Results do not depend on the order of the row lists (every point occurs at
// most once per item; all reductions run in a fixed order): deterministic.
#include "vlg_common.cuh"
#include "vlg_kernels.h"

namespace vlg {

namespace {

constexpr int NTHREADS = 256;
constexpr int DIFF_STRIDE = 52;  // floats per (m,row) Diff vector (X<=52; 16B rows)
constexpr int BS_FLOATS = 16 * 128;

// transposed + swizzled activation tile: element (k, row)
__device__ __forceinline__ int as_idx(int k, int row) { return k * 128 + (row ^ (((k >> 2) & 7) << 2)); }

// column owned by (tx, j) in an NT=8 thread tile: two groups of 4 so B loads are 128-bit
// and conflict free.
__device__ __forceinline__ int col8(int tx, int j) { return j < 4 ? 4 * tx + j : 64 + 4 * tx + (j - 4); }

// acc[8][NT] += A(128 x Kdim, in As) * B(Kdim x 16*NT, rows of Bg in global/L2)
template <int NT>
__device__ __forceinline__ void gemm_tile(const float* __restrict__ As, float* __restrict__ Bs,
                                          const float* __restrict__ Bg, int Kdim, float (&acc)[8][NT]) {
  constexpr int N = 16 * NT;
  constexpr int F4 = 16 * N / 4;          // float4 per 16-row slab
  constexpr int LD = F4 / NTHREADS;       // 2 (N=128) or 1 (N=64)
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int nchunks = Kdim / 16;
  float4 pre[LD];
  const float4* Bg4 = reinterpret_cast<const float4*>(Bg);
#pragma unroll
  for (int i = 0; i < LD; ++i) pre[i] = __ldg(Bg4 + tid + i * NTHREADS);
#pragma unroll
  for (int i = 0; i < LD; ++i) reinterpret_cast<float4*>(Bs)[tid + i * NTHREADS] = pre[i];
  __syncthreads();
  for (int c = 0; c < nchunks; ++c) {
    if (c + 1 < nchunks) {
#pragma unroll
      for (int i = 0; i < LD; ++i) pre[i] = __ldg(Bg4 + (c + 1) * F4 + tid + i * NTHREADS);
    }
    const float* B = Bs + (c & 1) * BS_FLOATS;
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      const int k = c * 16 + kk;
      float4 a0 = *reinterpret_cast<const float4*>(As + as_idx(k, 8 * ty));
      float4 a1 = *reinterpret_cast<const float4*>(As + as_idx(k, 8 * ty + 4));
      float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      float bv[NT];
      float4 b0 = *reinterpret_cast<const float4*>(B + kk * N + 4 * tx);
      bv[0] = b0.x; bv[1] = b0.y; bv[2] = b0.z; bv[3] = b0.w;
      if constexpr (NT == 8) {
        float4 b1 = *reinterpret_cast<const float4*>(B + kk * N + 64 + 4 * tx);
        bv[4] = b1.x; bv[5] = b1.y; bv[6] = b1.z; bv[7] = b1.w;
      }
      // packed f32x2 FMAs (two independent IEEE fmas per instruction: same bits as scalar fmaf, half the issue slots)
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float2 a2 = make_float2(av[i], av[i]);
#pragma unroll
        for (int j = 0; j < NT; j += 2) {
          const float2 r = __ffma2_rn(a2, make_float2(bv[j], bv[j + 1]), make_float2(acc[i][j], acc[i][j + 1]));
          acc[i][j] = r.x;
          acc[i][j + 1] = r.y;
        }
      }
    }
    if (c + 1 < nchunks) {
      float4* dst = reinterpret_cast<float4*>(Bs + ((c + 1) & 1) * BS_FLOATS);
#pragma unroll
      for (int i = 0; i < LD; ++i) dst[tid + i * NTHREADS] = pre[i];
    }
    __syncthreads();
  }
}

// write a thread's 8x8 accumulator tile transposed into As (kk = column)
__device__ __forceinline__ void store_tile_T(float* As, const float (&acc)[8][8]) {
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int c = col8(tx, j);
    *reinterpret_cast<float4*>(As + as_idx(c, 8 * ty)) = make_float4(acc[0][j], acc[1][j], acc[2][j], acc[3][j]);
    *reinterpret_cast<float4*>(As + as_idx(c, 8 * ty + 4)) = make_float4(acc[4][j], acc[5][j], acc[6][j], acc[7][j]);
  }
}

__device__ __forceinline__ float pre1(const float* sw, int c, float2 z) {
  // first-layer pre-activation; the same expression is used in forward and backward so
  // the recomputed ReLU mask is bit-identical.
  return fmaf(sw[OFF_W1Y + c], z.y, fmaf(sw[OFF_W1X + c], z.x, sw[OFF_B1 + c]));
}

constexpr int SIMT_MAX_W = 512;   // points per window
constexpr int SIMT_MAX_ITEMS = 288;  // >= K + 2*M*W/128 + 1 for K <= 254, M <= 4, W <= 512 ... checked on the host

struct Smem {
  float* As;       // 128*128
  float* Bs;       // 2*16*128
  float* sw;       // 576 small weights of the current decoder
  float* coef;     // 64
  float* basis;    // 32*9
  float* om;       // 18 omega, 18 m, 18 v
  float* gacc;     // 18
  float* red;      // 8*20
  int* cnt;        // 256
  uint16_t* item;  // SIMT_MAX_ITEMS: decoder | tile << 8
  float* Diff;     // M*W*52
  float2* zs;      // W
  float2* dzs;     // W
  float* ts;       // W
  uint8_t* sel;    // MAX_M*2*W
  uint16_t* rows;  // K*W
};

constexpr int SFIX = 128 * 128 + 2 * BS_FLOATS + 576 + 64 + 4 * MAX_NPOLY * MAX_KB + (3 * 2 * MAX_KB + 2) +
                     (2 * MAX_KB + 2) + 8 * 20 + 256 + SIMT_MAX_ITEMS / 2;

__device__ __forceinline__ Smem carve(unsigned char* base, int M, int W) {
  Smem s;
  float* f = reinterpret_cast<float*>(base);
  s.As = f; f += 128 * 128;
  s.Bs = f; f += 2 * BS_FLOATS;
  s.sw = f; f += 576;
  s.coef = f; f += 64;
  s.basis = f; f += 4 * MAX_NPOLY * MAX_KB;
  s.om = f; f += 3 * 2 * MAX_KB + 2;
  s.gacc = f; f += 2 * MAX_KB + 2;
  s.red = f; f += 8 * 20;
  s.cnt = reinterpret_cast<int*>(f); f += 256;
  s.item = reinterpret_cast<uint16_t*>(f); f += SIMT_MAX_ITEMS / 2;
  s.Diff = f; f += M * W * DIFF_STRIDE;
  s.zs = reinterpret_cast<float2*>(f); f += 2 * W;
  s.dzs = reinterpret_cast<float2*>(f); f += 2 * W;
  s.ts = f; f += W;
  s.sel = reinterpret_cast<uint8_t*>(f); f += MAX_M * 2 * W / 4 + 1;
  s.rows = reinterpret_cast<uint16_t*>(f);
  return s;
}

}  // namespace

static size_t simt_smem_bytes_w(int W, int K, int M) {
  size_t fl = size_t(SFIX) + size_t(M) * W * DIFF_STRIDE + 2 * size_t(W) + 2 * size_t(W) + W + MAX_M * 2 * size_t(W) / 4 + 1;
  return fl * 4 + size_t(K) * W * 2 + 16;
}
static int simt_max_items(int W, int K, int M) { return K + 2 * M * W / 128 + 1; }

// Window length: fewest 128-row items per curve under the shared-memory budget (same expected-cost
// model as the tensor-core kernel: a decoder is drawn by a point with probability 1-(1-1/K)^(2M)).
static int simt_window_points(int T, int K, int M) {
  const double p = 1.0 - pow(1.0 - 1.0 / K, 2.0 * M);
  const int segs = T - 1;
  int best_w = 0;
  double best = 1e300;
  for (int nwin = 1; nwin <= segs; ++nwin) {
    const int w = (segs + nwin - 1) / nwin + 1;
    if (w <= SIMT_MAX_W && simt_smem_bytes_w(w, K, M) <= 232448 && simt_max_items(w, K, M) <= SIMT_MAX_ITEMS) {
      const double cost = nwin * (K * expected_items(w, p) + 0.25);
      if (cost < best) { best = cost; best_w = w; }
    }
    if (w <= 128) break;
  }
  return best_w;  // 0: does not fit
}
// layer-2 ReLU mask bits [cta][item][128 rows][16 bytes], L2 resident
size_t simt_workspace_bytes(int N, int T, int K, int M) {
  const int W = simt_window_points(T, K, M);
  if (W == 0) return 0;
  return 256 + size_t(persistent_grid(N)) * simt_max_items(W, K, M) * 2048;   // 256-byte header: word [1] = status flags
}

template <StepMode MODE>
__global__ void __launch_bounds__(NTHREADS, 1) simt_curve_kernel(StepParams p, int W, int max_items) {
  constexpr bool GRAD = MODE != StepMode::Energy;       // backward items
  constexpr bool GOUT = MODE == StepMode::EnergyGrad;   // gradient out instead of Adam
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4, lane = tid & 31, warp = tid >> 5;
  const int M = p.M, K = p.K, T = p.T, n_poly = p.n_poly, Kb = p.Kb, X = p.X;
  Smem s = carve(smem_raw, M, W);
  unsigned int* status = reinterpret_cast<unsigned int*>(p.workspace) + 1;   // VLG_STATUS_* flags (header zeroed by the launcher)
  uint8_t* mask2 = reinterpret_cast<uint8_t*>(p.workspace) + 256 + size_t(blockIdx.x) * max_items * 2048;
  bool bad_draw = false;
  if (blockIdx.x == 0 && tid == 0 && !packed_header_ok(p.packed, p.K_total, p.X)) atomicOr(status, unsigned(VLG_STATUS_BAD_PACKED));
  const int WSEG = W - 1;
  const int nwin = (T - 1 + WSEG - 1) / WSEG;
  // gradient-output mode: dE/da, dE/db accumulate in the Adam-moment slots of s.om, which this mode does not use
  float* gab = s.om + 2 * MAX_KB;
  for (int i = tid; i < 4 * n_poly * Kb; i += NTHREADS) s.basis[i] = p.basis[i];

  for (int n = blockIdx.x; n < p.N; n += gridDim.x) {
  // ---- per-curve state -> shared ----
  if (tid < 2 * Kb) {
    s.om[tid] = p.omega[size_t(n) * 2 * Kb + tid];
    if (MODE == StepMode::Optimize) {
      s.om[2 * MAX_KB + tid] = p.adam_m[size_t(n) * 2 * Kb + tid];
      s.om[4 * MAX_KB + tid] = p.adam_v[size_t(n) * 2 * Kb + tid];
    }
  }
  const float2 pa = make_float2(p.a[2 * n], p.a[2 * n + 1]);
  const float2 pb = make_float2(p.b[2 * n], p.b[2 * n + 1]);
  const int dec_base = curve_dec_base(p, n, tid == 0, status);
  const float coefm = 2.0f / float(M);
  __syncthreads();

  for (int step = 0; step < p.steps; ++step) {
    // coef = basis @ omega  [n_poly][4][2]
    if (tid < 8 * n_poly) {
      const int r = tid >> 1, d = tid & 1;
      float acc = 0.f;
      for (int k = 0; k < Kb; ++k) acc = fmaf(s.basis[r * Kb + k], s.om[2 * k + d], acc);
      s.coef[tid] = acc;
    }
    if (tid < 2 * MAX_KB) s.gacc[tid] = 0.f;
    if (GOUT && tid < 4) gab[tid] = 0.f;
    float e_tot = 0.f, l_tot = 0.f;  // meaningful in thread 0
    __syncthreads();

    for (int win = 0; win < nwin; ++win) {
      const int seg0 = win * WSEG;
      const int nseg = min(WSEG, T - 1 - seg0);
      // ---- window setup: points, draws, clear accumulators ----
      for (int pt = tid; pt < W; pt += NTHREADS) {
        const int ti = min(seg0 + pt, T - 1);
        const float t = p.t[ti];
        s.ts[pt] = t;
        s.zs[pt] = spline_point(t, n_poly, s.coef, pa, pb);
        s.dzs[pt] = make_float2(0.f, 0.f);
        if (p.draws != nullptr) {
          for (int m = 0; m < M; ++m)
            for (int role = 0; role < 2; ++role) {
              s.sel[(m * 2 + role) * W + pt] = pt < nseg ? explicit_draw(p.draws, p.steps, M, T, K, n, step, m, role, seg0 + pt, bad_draw) : 255;
            }
        } else {
          for (int jp = 0; jp < (M + 1) / 2; ++jp) {
            uint32_t d[4] = {255u, 255u, 255u, 255u};
            if (pt < nseg)
              counter_draws4(p.seed, uint32_t(p.curve_id0 + n), uint32_t(p.step0 + step), uint32_t(seg0 + pt),
                             uint32_t(jp), uint32_t(K), d);
            for (int q = 0; q < 4; ++q) {
              const int m = 2 * jp + (q >> 1);
              if (m < M) s.sel[(m * 2 + (q & 1)) * W + pt] = uint8_t(d[q]);
            }
          }
        }
      }
      for (int i = tid; i < M * W * DIFF_STRIDE / 4; i += NTHREADS)
        reinterpret_cast<float4*>(s.Diff)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int i = tid; i < K; i += NTHREADS) s.cnt[i] = 0;
      __syncthreads();
      // ---- per-decoder row lists: the points of the window that drew decoder k ----
      for (int pt = tid; pt <= nseg; pt += NTHREADS) {
        int cand[2 * MAX_M];
        int nc = 0;
        for (int m = 0; m < M; ++m) {
          if (pt < nseg) cand[nc++] = s.sel[(m * 2 + 0) * W + pt];
          if (pt >= 1) cand[nc++] = s.sel[(m * 2 + 1) * W + pt - 1];
        }
        for (int i = 0; i < nc; ++i) {
          bool dup = false;
          for (int j = 0; j < i; ++j) dup |= (cand[j] == cand[i]);
          if (!dup) {
            const int slot = atomicAdd(&s.cnt[cand[i]], 1);
            s.rows[cand[i] * W + slot] = uint16_t(pt);
          }
        }
      }
      __syncthreads();
      if (tid == 0) {
        int ni = 0;
        for (int k = 0; k < K; ++k)
          for (int q = 0; q * 128 < s.cnt[k]; ++q) s.item[ni++] = uint16_t(k | (q << 8));
        s.red[159] = __int_as_float(ni);
      }
      __syncthreads();
      const int nitems = __float_as_int(s.red[159]);

      // =============================== forward ===============================
      for (int it = 0; it < nitems; ++it) {
        const int k = s.item[it] & 0xFF, q0 = (s.item[it] >> 8) * 128;
        const int nrows = min(128, s.cnt[k] - q0);
        const uint16_t* rl = s.rows + k * W + q0;
        const float* dec = dec_ptr(p.packed, dec_base + k);
        for (int i = tid; i < 576; i += NTHREADS) s.sw[i] = __ldg(dec + i);
        __syncthreads();
        {  // layer 1 on CUDA cores -> As[c][row]
          const int row = tid & 127, c0 = (tid >> 7) * 64;
          const float2 z = s.zs[row < nrows ? rl[row] : 0];
#pragma unroll 8
          for (int c = c0; c < c0 + 64; ++c) s.As[as_idx(c, row)] = fmaxf(pre1(s.sw, c, z), 0.f);
        }
        __syncthreads();
        {  // layer 2: h2 = relu(h1 W2^T + b2), mask bits
          float acc[8][8];
#pragma unroll
          for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
          gemm_tile<8>(s.As, s.Bs, dec + OFF_W2T, H, acc);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            uint32_t bits = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float v = acc[i][j] + s.sw[OFF_B2 + col8(tx, j)];
              if (v > 0.f) bits |= 1u << j;
              acc[i][j] = fmaxf(v, 0.f);
            }
            if (GRAD) mask2[(size_t(it) * 128 + 8 * ty + i) * 16 + tx] = uint8_t(bits);
          }
          store_tile_T(s.As, acc);  // gemm_tile ended with a barrier: As is free
        }
        __syncthreads();
        {  // layer 3: x = h2 W3^T + b3 -> Diff
          float acc[8][4];
#pragma unroll
          for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
          gemm_tile<4>(s.As, s.Bs, dec + OFF_W3T, H, acc);
          const int c = 4 * tx;
          int pts[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) pts[i] = (8 * ty + i < nrows) ? int(rl[8 * ty + i]) : -1;
          if (c < X) {
            float4 bb = *reinterpret_cast<const float4*>(s.sw + OFF_B3 + c);
            // role 0: this point is the left end of its segment
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int pt = pts[i];
              acc[i][0] += bb.x; acc[i][1] += bb.y; acc[i][2] += bb.z; acc[i][3] += bb.w;
              if (pt < 0) continue;
              for (int m = 0; m < M; ++m)
                if (s.sel[(m * 2 + 0) * W + pt] == k) {
                  float4* d = reinterpret_cast<float4*>(s.Diff + (m * W + pt) * DIFF_STRIDE + c);
                  float4 v = *d;
                  v.x -= acc[i][0]; v.y -= acc[i][1]; v.z -= acc[i][2]; v.w -= acc[i][3];
                  *d = v;
                }
            }
          }
          __syncthreads();
          if (c < X) {
            // role 1: this point is the right end of the previous segment
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int pt = pts[i];
              if (pt < 1) continue;
              for (int m = 0; m < M; ++m)
                if (s.sel[(m * 2 + 1) * W + pt - 1] == k) {
                  float4* d = reinterpret_cast<float4*>(s.Diff + (m * W + pt - 1) * DIFF_STRIDE + c);
                  float4 v = *d;
                  v.x += acc[i][0]; v.y += acc[i][1]; v.z += acc[i][2]; v.w += acc[i][3];
                  *d = v;
                }
            }
          }
        }
        __syncthreads();
      }

      // =============================== energy ===============================
      {
        float e = 0.f, l = 0.f;
        for (int m = 0; m < M; ++m)
          for (int r = tid; r < nseg; r += NTHREADS) {
            const float* d = s.Diff + (m * W + r) * DIFF_STRIDE;
            float q = 0.f;
            for (int c = 0; c < X; ++c) q = fmaf(d[c], d[c], q);
            e += q;
            l += sqrtf(q);
          }
        e = warp_sum(e);
        l = warp_sum(l);
        if (lane == 0) { s.red[warp] = e; s.red[8 + warp] = l; }
        __syncthreads();
        if (tid == 0) {
          float ee = 0.f, ll = 0.f;
          for (int w = 0; w < 8; ++w) { ee += s.red[w]; ll += s.red[8 + w]; }
          e_tot += ee;
          l_tot += ll;
        }
        __syncthreads();
      }

      if (GRAD) {
        // =============================== backward ===============================
        for (int it = 0; it < nitems; ++it) {
          const int k = s.item[it] & 0xFF, q0 = (s.item[it] >> 8) * 128;
          const int nrows = min(128, s.cnt[k] - q0);
          const uint16_t* rl = s.rows + k * W + q0;
          const float* dec = dec_ptr(p.packed, dec_base + k);
          for (int i = tid; i < 576; i += NTHREADS) s.sw[i] = __ldg(dec + i);
          {  // G = dE/dx_k  -> As[c][row], c < 64
            const int row = tid & 127, c0 = (tid >> 7) * 32;
            const int pt = row < nrows ? int(rl[row]) : -1;
            float g[32];
#pragma unroll
            for (int c = 0; c < 32; ++c) g[c] = 0.f;
            for (int m = 0; m < (pt >= 0 ? M : 0); ++m) {
              if (pt >= 1 && s.sel[(m * 2 + 1) * W + pt - 1] == k) {
                const float* d = s.Diff + (m * W + pt - 1) * DIFF_STRIDE;
#pragma unroll
                for (int c = 0; c < 32; ++c)
                  if (c0 + c < X) g[c] += d[c0 + c];
              }
              if (s.sel[(m * 2 + 0) * W + pt] == k) {
                const float* d = s.Diff + (m * W + pt) * DIFF_STRIDE;
#pragma unroll
                for (int c = 0; c < 32; ++c)
                  if (c0 + c < X) g[c] -= d[c0 + c];
              }
            }
#pragma unroll
            for (int c = 0; c < 32; ++c) s.As[as_idx(c0 + c, row)] = coefm * g[c];
          }
          __syncthreads();
          float acc[8][8];
#pragma unroll
          for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
          gemm_tile<8>(s.As, s.Bs, dec + OFF_W3, XP, acc);  // dh2 = G W3
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const uint32_t bits = mask2[(size_t(it) * 128 + 8 * ty + i) * 16 + tx];
#pragma unroll
            for (int j = 0; j < 8; ++j)
              if (!((bits >> j) & 1u)) acc[i][j] = 0.f;
          }
          store_tile_T(s.As, acc);
          __syncthreads();
#pragma unroll
          for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
          gemm_tile<8>(s.As, s.Bs, dec + OFF_W2, H, acc);  // dh1 = dh2 W2
          // layer-1 mask (recomputed) and dz = dh1 W1, reduced over the 16 column threads
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int r = 8 * ty + i;
            const int pt = r < nrows ? int(rl[r]) : -1;     // uniform over the 16 column threads of the row
            const float2 z = s.zs[pt < 0 ? 0 : pt];
            float dx = 0.f, dy = 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int c = col8(tx, j);
              if (pre1(s.sw, c, z) > 0.f) {
                dx = fmaf(acc[i][j], s.sw[OFF_W1X + c], dx);
                dy = fmaf(acc[i][j], s.sw[OFF_W1Y + c], dy);
              }
            }
#pragma unroll
            for (int o = 8; o > 0; o >>= 1) {
              dx += __shfl_xor_sync(0xffffffffu, dx, o);
              dy += __shfl_xor_sync(0xffffffffu, dy, o);
            }
            // a point occurs at most once per item and items run one after the other: plain read-modify-write
            if (tx == 0 && pt >= 0) {
              float2 d = s.dzs[pt];
              d.x += dx;
              d.y += dy;
              s.dzs[pt] = d;
            }
          }
          __syncthreads();
        }
        // ---- d(omega) += P^T dz over the points of the window ----
        for (int base = 0; base < W; base += NTHREADS) {
          const int pt = base + tid;
          float P[MAX_KB];
          float2 dz = make_float2(0.f, 0.f);
          float tp = 0.f;
          if (pt < W) {
            tp = s.ts[pt];
            design_row(tp, n_poly, Kb, s.basis, P);
            dz = s.dzs[pt];
          } else {
#pragma unroll
            for (int k = 0; k < MAX_KB; ++k) P[k] = 0.f;
          }
#pragma unroll
          for (int k = 0; k < MAX_KB; ++k)
            if (k < Kb) {
              float cx = warp_sum(P[k] * dz.x), cy = warp_sum(P[k] * dz.y);
              if (lane == 0) { s.red[warp * 20 + 2 * k] = cx; s.red[warp * 20 + 2 * k + 1] = cy; }
            }
          __syncthreads();
          if (tid < 2 * Kb) {
            float g = 0.f;
            for (int w = 0; w < 8; ++w) g += s.red[w * 20 + tid];
            s.gacc[tid] += g;
          }
          __syncthreads();
          if (GOUT) {   // dE/da += sum (1-t) dz, dE/db += sum t dz: the design row extended by (1-t, t), second pass
            const float ax = warp_sum((1.0f - tp) * dz.x), ay = warp_sum((1.0f - tp) * dz.y);
            const float bx = warp_sum(tp * dz.x), by = warp_sum(tp * dz.y);
            if (lane == 0) { s.red[warp * 20] = ax; s.red[warp * 20 + 1] = ay; s.red[warp * 20 + 2] = bx; s.red[warp * 20 + 3] = by; }
            __syncthreads();
            if (tid < 4) {
              float g = 0.f;
              for (int w = 0; w < 8; ++w) g += s.red[w * 20 + tid];
              gab[tid] += g;
            }
            __syncthreads();
          }
        }
      }
    }  // windows

    // ---- step epilogue: energy out; gradient out, or penalty gradient and Adam ----
    if (tid == 0) write_energy(p, n, step, e_tot, l_tot, status);
    if (GOUT && tid < 2 * Kb + 4) write_grad(p, n, tid, tid < 2 * Kb ? s.gacc[tid] : gab[tid - 2 * Kb], status);
    if (MODE == StepMode::Optimize && tid < 2 * Kb) penalty_adam_step(p, step, tid, s.gacc[tid], s.basis, s.coef, pa, pb, s.om);
    __syncthreads();
  }  // steps

  if (MODE == StepMode::Optimize && tid < 2 * Kb) write_back(p, n, tid, s.om, status);
  __syncthreads();
  }  // curves of this CTA
  if (bad_draw) atomicOr(status, unsigned(VLG_STATUS_BAD_DRAW));
}

cudaError_t launch_simt(const StepParams& p, cudaStream_t stream) {
  const int W = simt_window_points(p.T, p.K, p.M);
  if (W < 2) return cudaErrorNotSupported;
  const size_t smem = simt_smem_bytes_w(W, p.K, p.M);
  const int grid = persistent_grid(p.N);
  const int max_items = simt_max_items(W, p.K, p.M);
  if (p.workspace == nullptr || p.workspace_bytes < simt_workspace_bytes(p.N, p.T, p.K, p.M)) return cudaErrorInvalidValue;
  cudaError_t e = cudaMemsetAsync(p.workspace, 0, 256, stream);
  if (e != cudaSuccess) return e;
  auto launch = [&](auto kernel) -> cudaError_t {
    cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (err != cudaSuccess) return err;
    kernel<<<grid, NTHREADS, smem, stream>>>(p, W, max_items);
    return cudaGetLastError();
  };
  return with_mode(p.mode, [&](auto mode) { return launch(simt_curve_kernel<decltype(mode)::value>); });
}

}  // namespace vlg
