// Weight repacking and the small helpers (disagreement field, spline evaluation and its
// backward, least-squares spline fit).  None of these are hot; they exist so the
// drop-in entry points never leave the GPU and never need a CPU fallback.
#include <cuda_fp16.h>

#include "vlg_common.cuh"
#include "vlg_kernels.h"

namespace vlg {

namespace {

__device__ __forceinline__ float tf32_rn(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

// one block per decoder
__global__ void pack_kernel(const float* __restrict__ W1, const float* __restrict__ b1,
                            const float* __restrict__ W2, const float* __restrict__ b2,
                            const float* __restrict__ W3, const float* __restrict__ b3, int K, int X,
                            void* packed) {
  const int k = blockIdx.x;
  if (k == 0 && threadIdx.x == 0) {
    PackedHeader* h = reinterpret_cast<PackedHeader*>(packed);
    h->magic = PACK_MAGIC;
    h->K = K;
    h->Hdim = H;
    h->X = X;
    h->dec_floats = DEC_FLOATS;
  }
  float* d = const_cast<float*>(dec_ptr(packed, k));
  const float* w1 = W1 + size_t(k) * H * 2;
  const float* w2 = W2 + size_t(k) * H * H;
  const float* w3 = W3 + size_t(k) * X * H;
  for (int i = threadIdx.x; i < 256; i += blockDim.x) d[((i & 1) ? OFF_W1Y : OFF_W1X) + (i >> 1)] = w1[i];
  for (int i = threadIdx.x; i < H; i += blockDim.x) {
    d[OFF_B1 + i] = b1[size_t(k) * H + i];
    d[OFF_B2 + i] = b2[size_t(k) * H + i];
  }
  for (int i = threadIdx.x; i < XP; i += blockDim.x) d[OFF_B3 + i] = i < X ? b3[size_t(k) * X + i] : 0.f;
  for (int i = threadIdx.x; i < H * H; i += blockDim.x) {
    const int o = i / H, in = i % H;  // W2[o][in]
    const float w = w2[i];
    d[OFF_W2 + i] = w;
    d[OFF_W2T + in * H + o] = w;
    const int u = ((in >> 2) * H + o) * 4 + (in & 3);   // B[n=o][k=in]
    const int ut = ((o >> 2) * H + in) * 4 + (o & 3);   // B[n=in][k=o]
    const float hi = tf32_rn(w);
    d[OFF_W2_UMMA + u] = hi;
    d[OFF_W2T_UMMA + ut] = hi;
    const __half wh = __float2half_rn(w);
    const __half wl = __float2half_rn(w - __half2float(wh));
    reinterpret_cast<__half*>(d + OFF_W2_H)[((in >> 3) * H + o) * 8 + (in & 7)] = wh;
    reinterpret_cast<__half*>(d + OFF_W2T_H)[((o >> 3) * H + in) * 8 + (o & 7)] = wh;
    reinterpret_cast<__half*>(d + OFF_W2_HL)[((in >> 3) * H + o) * 8 + (in & 7)] = wl;
    reinterpret_cast<__half*>(d + OFF_W2T_HL)[((o >> 3) * H + in) * 8 + (o & 7)] = wl;
  }
  for (int i = threadIdx.x; i < XP * H; i += blockDim.x) {
    const int o = i / H, in = i % H;  // W3[o][in], zero rows o >= X
    const float w = o < X ? w3[o * H + in] : 0.f;
    d[OFF_W3 + i] = w;
    d[OFF_W3T + in * XP + o] = w;
    const int u = ((in >> 2) * XP + o) * 4 + (in & 3);   // B[n=o][k=in], N = 64
    const int ut = ((o >> 2) * H + in) * 4 + (o & 3);    // B[n=in][k=o], N = 128, K = 64
    const float hi = tf32_rn(w);
    d[OFF_W3_UMMA + u] = hi;
    d[OFF_W3T_UMMA + ut] = hi;
    const __half wh = __float2half_rn(w);
    const __half wl = __float2half_rn(w - __half2float(wh));
    reinterpret_cast<__half*>(d + OFF_W3_H)[((in >> 3) * XP + o) * 8 + (in & 7)] = wh;   // N = 64, K = 128
    reinterpret_cast<__half*>(d + OFF_W3T_H)[((o >> 3) * H + in) * 8 + (o & 7)] = wh;    // N = 128, K = 64
    reinterpret_cast<__half*>(d + OFF_W3_HL)[((in >> 3) * XP + o) * 8 + (in & 7)] = wl;
    reinterpret_cast<__half*>(d + OFF_W3T_HL)[((o >> 3) * H + in) * 8 + (o & 7)] = wl;
  }
}

// ---- ensemble disagreement field (src/init_splines_ensemble.py:49-51) ----
// block = 128 threads, 32 grid points; thread j owns hidden unit j (layers 1,2) and
// output o=j (layer 3, j<64) for all 32 points; Welford over decoders.
constexpr int SP = 32;
__global__ void __launch_bounds__(128) std_norm_kernel(const void* packed, int K, int X, int G,
                                                        const float* __restrict__ grid, float* __restrict__ out) {
  __shared__ float h1[SP][H + 1];
  __shared__ float h2[SP][H + 1];
  __shared__ float zz[SP][2];
  __shared__ float red[SP][4];
  const int j = threadIdx.x, g0 = blockIdx.x * SP;
  if (j < SP * 2) {
    const int p = j >> 1, gi = min(g0 + p, G - 1);
    zz[p][j & 1] = grid[2 * gi + (j & 1)];
  }
  float mean[SP], m2[SP];
#pragma unroll
  for (int p = 0; p < SP; ++p) mean[p] = m2[p] = 0.f;
  __syncthreads();
  for (int k = 0; k < K; ++k) {
    const float* d = dec_ptr(packed, k);
    {
      const float wa = d[OFF_W1X + j], wb = d[OFF_W1Y + j], bb = d[OFF_B1 + j];
#pragma unroll
      for (int p = 0; p < SP; ++p) h1[p][j] = fmaxf(fmaf(wb, zz[p][1], fmaf(wa, zz[p][0], bb)), 0.f);
    }
    __syncthreads();
    {
      float acc[SP];
      const float bb = d[OFF_B2 + j];
#pragma unroll
      for (int p = 0; p < SP; ++p) acc[p] = bb;
      for (int i = 0; i < H; ++i) {
        const float w = __ldg(d + OFF_W2T + i * H + j);
#pragma unroll
        for (int p = 0; p < SP; ++p) acc[p] = fmaf(h1[p][i], w, acc[p]);
      }
#pragma unroll
      for (int p = 0; p < SP; ++p) h2[p][j] = fmaxf(acc[p], 0.f);
    }
    __syncthreads();
    if (j < XP) {
      float acc[SP];
      const float bb = d[OFF_B3 + j];
#pragma unroll
      for (int p = 0; p < SP; ++p) acc[p] = bb;
      for (int i = 0; i < H; ++i) {
        const float w = __ldg(d + OFF_W3T + i * XP + j);
#pragma unroll
        for (int p = 0; p < SP; ++p) acc[p] = fmaf(h2[p][i], w, acc[p]);
      }
      const float inv = 1.0f / float(k + 1);
#pragma unroll
      for (int p = 0; p < SP; ++p) {
        const float dl = acc[p] - mean[p];
        mean[p] += dl * inv;
        m2[p] = fmaf(dl, acc[p] - mean[p], m2[p]);
      }
    }
    __syncthreads();
  }
  // sum of variances over the X outputs (threads 0..X-1), then sqrt
  const float invk = K > 1 ? 1.0f / float(K - 1) : 0.f;
#pragma unroll
  for (int p = 0; p < SP; ++p) {
    float v = (j < X) ? m2[p] * invk : 0.f;
    v = warp_sum(v);
    if ((j & 31) == 0) red[p][j >> 5] = v;
  }
  __syncthreads();
  if (j < SP && g0 + j < G) out[g0 + j] = sqrtf((red[j][0] + red[j][1]) + (red[j][2] + red[j][3]));
}

__global__ void spline_points_kernel(int N, int T, int n_poly, const float* __restrict__ a,
                                     const float* __restrict__ b, const float* __restrict__ omega,
                                     const float* __restrict__ basis, const float* __restrict__ t,
                                     float* __restrict__ z) {
  __shared__ float coef[MAX_NPOLY * 8];
  const int n = blockIdx.x, Kb = n_poly + 1;
  if (threadIdx.x < 8 * n_poly) {
    const int r = threadIdx.x >> 1, d = threadIdx.x & 1;
    float acc = 0.f;
    for (int k = 0; k < Kb; ++k) acc = fmaf(basis[r * Kb + k], omega[(size_t(n) * Kb + k) * 2 + d], acc);
    coef[threadIdx.x] = acc;
  }
  __syncthreads();
  const float2 pa = make_float2(a[2 * n], a[2 * n + 1]), pb = make_float2(b[2 * n], b[2 * n + 1]);
  for (int i = threadIdx.x; i < T; i += blockDim.x) {
    float2 zz = spline_point(t[i], n_poly, coef, pa, pb);
    z[(size_t(i) * N + n) * 2] = zz.x;
    z[(size_t(i) * N + n) * 2 + 1] = zz.y;
  }
}

// Backward of spline_points_kernel: z[t] = (1-t) a + t b + P[t] omega is linear in (omega, a, b), so
// d(omega) = sum_t P[t]^T dz[t], da = sum_t (1-t) dz[t], db = sum_t t dz[t].  One block per curve; each thread sums
// its points in order, then the warps and the block reduce in a fixed order: repeated calls give the same bits.
__global__ void __launch_bounds__(256) spline_points_backward_kernel(int N, int T, int n_poly,
                                                                     const float* __restrict__ basis,
                                                                     const float* __restrict__ t,
                                                                     const float* __restrict__ dz,
                                                                     float* __restrict__ grad_omega,
                                                                     float* __restrict__ grad_a,
                                                                     float* __restrict__ grad_b) {
  constexpr int NCOL = 2 * MAX_KB + 4;   // 2 Kb columns of P^T dz, then (1-t) dz and t dz
  __shared__ float red[8][NCOL];
  const int n = blockIdx.x, Kb = n_poly + 1, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float acc[NCOL];
#pragma unroll
  for (int c = 0; c < NCOL; ++c) acc[c] = 0.f;
  for (int i = threadIdx.x; i < T; i += blockDim.x) {
    const float ti = t[i];
    const float dx = dz[(size_t(i) * N + n) * 2], dy = dz[(size_t(i) * N + n) * 2 + 1];
    float P[MAX_KB];
    design_row(ti, n_poly, Kb, basis, P);
#pragma unroll
    for (int k = 0; k < MAX_KB; ++k)
      if (k < Kb) {
        acc[2 * k] = fmaf(P[k], dx, acc[2 * k]);
        acc[2 * k + 1] = fmaf(P[k], dy, acc[2 * k + 1]);
      }
    acc[NCOL - 4] = fmaf(1.0f - ti, dx, acc[NCOL - 4]);
    acc[NCOL - 3] = fmaf(1.0f - ti, dy, acc[NCOL - 3]);
    acc[NCOL - 2] = fmaf(ti, dx, acc[NCOL - 2]);
    acc[NCOL - 1] = fmaf(ti, dy, acc[NCOL - 1]);
  }
#pragma unroll
  for (int c = 0; c < NCOL; ++c) {
    const float v = warp_sum(acc[c]);
    if (lane == 0) red[warp][c] = v;
  }
  __syncthreads();
  const int c = threadIdx.x;
  if (c < NCOL && (c < 2 * Kb || c >= NCOL - 4)) {
    float g = 0.f;
    for (int w = 0; w < 8; ++w) g += red[w][c];
    if (c < 2 * Kb) grad_omega[size_t(n) * 2 * Kb + c] = g;
    else if (c < NCOL - 2) grad_a[2 * n + c - (NCOL - 4)] = g;
    else grad_b[2 * n + c - (NCOL - 2)] = g;
  }
}

// ---- least-squares fit of the spline to a poly-line (init_splines_ensemble.py:172-193) ----
// one warp per curve; normal equations in double, Gaussian elimination with pivoting.
__global__ void __launch_bounds__(32) fit_splines_kernel(int N, int Lmax, int n_poly,
                                                         const float* __restrict__ targets,
                                                         const int32_t* __restrict__ lens,
                                                         const float* __restrict__ basis, float* __restrict__ omega,
                                                         float* __restrict__ ab) {
  const int n = blockIdx.x, lane = threadIdx.x, Kb = n_poly + 1;
  const int L = lens[n];
  const float* tg = targets + size_t(n) * Lmax * 2;
  __shared__ double A[MAX_KB][MAX_KB + 2];
  const float ax = tg[0], ay = tg[1], bx = tg[2 * (L - 1)], by = tg[2 * (L - 1) + 1];
  double acc[MAX_KB * (MAX_KB + 1) / 2 + 2 * MAX_KB];
  for (int i = 0; i < MAX_KB * (MAX_KB + 1) / 2 + 2 * MAX_KB; ++i) acc[i] = 0.0;
  // torch.linspace(0,1,L) in fp32: symmetric formula (start + i*step | end - (L-1-i)*step)
  const float stepf = L > 1 ? 1.0f / float(L - 1) : 0.f;
  for (int i = lane; i < L; i += 32) {
    const float t = (i < L / 2) ? float(i) * stepf : 1.0f - float(L - 1 - i) * stepf;
    float P[MAX_KB];
    design_row(t, n_poly, Kb, basis, P);
    const double rx = double(tg[2 * i]) - (double(1.0f - t) * ax + double(t) * bx);
    const double ry = double(tg[2 * i + 1]) - (double(1.0f - t) * ay + double(t) * by);
    int q = 0;
    for (int r = 0; r < Kb; ++r)
      for (int c = r; c < Kb; ++c) acc[q++] += double(P[r]) * double(P[c]);
    for (int r = 0; r < Kb; ++r) {
      acc[q++] += double(P[r]) * rx;
      acc[q++] += double(P[r]) * ry;
    }
  }
  const int nacc = Kb * (Kb + 1) / 2 + 2 * Kb;
  for (int i = 0; i < nacc; ++i)
    for (int o = 16; o > 0; o >>= 1) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], o);
  if (lane == 0) {
    int q = 0;
    for (int r = 0; r < Kb; ++r)
      for (int c = r; c < Kb; ++c) { A[r][c] = acc[q]; A[c][r] = acc[q]; ++q; }
    for (int r = 0; r < Kb; ++r) { A[r][Kb] = acc[q++]; A[r][Kb + 1] = acc[q++]; }
    // A path with fewer than Kb interior nodes leaves the normal equations rank deficient (every spline through
    // the nodes is optimal; the reference's LBFGS from omega = 0 lands near the minimum-norm one).  A ridge of
    // 1e-10 of the mean diagonal picks that solution and is far below fp32 resolution when the rank is full.
    double tr = 0.0;
    for (int r = 0; r < Kb; ++r) tr += A[r][r];
    const double ridge = 1e-10 * tr / double(Kb) + 1e-300;
    for (int r = 0; r < Kb; ++r) A[r][r] += ridge;
    for (int c = 0; c < Kb; ++c) {
      int piv = c;
      for (int r = c + 1; r < Kb; ++r) if (fabs(A[r][c]) > fabs(A[piv][c])) piv = r;
      if (piv != c) for (int j = 0; j < Kb + 2; ++j) { double tmp = A[c][j]; A[c][j] = A[piv][j]; A[piv][j] = tmp; }
      const double inv = A[c][c] != 0.0 ? 1.0 / A[c][c] : 0.0;
      for (int r = 0; r < Kb; ++r) {
        if (r == c) continue;
        const double f = A[r][c] * inv;
        for (int j = c; j < Kb + 2; ++j) A[r][j] -= f * A[c][j];
      }
    }
    for (int r = 0; r < Kb; ++r) {
      const double inv = A[r][r] != 0.0 ? 1.0 / A[r][r] : 0.0;
      omega[(size_t(n) * Kb + r) * 2] = float(A[r][Kb] * inv);
      omega[(size_t(n) * Kb + r) * 2 + 1] = float(A[r][Kb + 1] * inv);
    }
    ab[4 * n] = ax; ab[4 * n + 1] = ay; ab[4 * n + 2] = bx; ab[4 * n + 3] = by;
  }
}

}  // namespace

cudaError_t launch_pack(const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                        const float* b3, int K, int X, void* packed, cudaStream_t stream) {
  pack_kernel<<<K, 256, 0, stream>>>(W1, b1, W2, b2, W3, b3, K, X, packed);
  return cudaGetLastError();
}

cudaError_t launch_std_norm(const void* packed, int K, int X, int G, const float* grid, float* out,
                            cudaStream_t stream) {
  std_norm_kernel<<<(G + SP - 1) / SP, 128, 0, stream>>>(packed, K, X, G, grid, out);
  return cudaGetLastError();
}

cudaError_t launch_spline_points(int N, int T, int n_poly, const float* a, const float* b, const float* omega,
                                 const float* basis, const float* t, float* z, cudaStream_t stream) {
  spline_points_kernel<<<N, 256, 0, stream>>>(N, T, n_poly, a, b, omega, basis, t, z);
  return cudaGetLastError();
}

cudaError_t launch_spline_points_backward(int N, int T, int n_poly, const float* basis, const float* t, const float* dz,
                                          float* grad_omega, float* grad_a, float* grad_b, cudaStream_t stream) {
  spline_points_backward_kernel<<<N, 256, 0, stream>>>(N, T, n_poly, basis, t, dz, grad_omega, grad_a, grad_b);
  return cudaGetLastError();
}

cudaError_t launch_fit_splines(int N, int Lmax, int n_poly, const float* targets, const int32_t* lens,
                               const float* basis, float* omega, float* ab, cudaStream_t stream) {
  fit_splines_kernel<<<N, 32, 0, stream>>>(N, Lmax, n_poly, targets, lens, basis, omega, ab);
  return cudaGetLastError();
}

}  // namespace vlg
