// extern "C" front end: argument validation, device check, dispatch.  See include/vlg.h.
#include "../../include/vlg.h"

#include <limits.h>
#include <math.h>
#include <stdio.h>

#include "vlg_common.cuh"
#include "vlg_kernels.h"

namespace vlg {

int persistent_grid(int N) {
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0) sms = v;
  } else {
    (void)cudaGetLastError();
  }
  return N < sms ? N : sms;
}

double expected_items(int w, double p) {
  const double mean = w * p, sd = sqrt(w * p * (1.0 - p)) + 1e-9;
  double items = 0.0;
  for (int q = 0; q * 128 < w; ++q) items += 0.5 * erfc((q * 128 + 0.5 - mean) / (sd * 1.4142135623730951));  // P(n > 128 q)
  return items;
}

}  // namespace vlg

namespace {

thread_local char g_cuda_err[256] = "";

int cuda_fail(cudaError_t e) {
  snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", cudaGetErrorName(e), cudaGetErrorString(e));
  return VLG_ERR_CUDA;
}

int check_device() {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return cuda_fail(e);
  int major = 0;
  e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e != cudaSuccess) return cuda_fail(e);
  if (major != 10) return VLG_ERR_DEVICE;
  return VLG_OK;
}

// What the three step entry points share: the device check, the shape and workspace checks, the fields every mode
// sets, and the launch of the fp32 or the tensor-core kernel.  `p` comes with the mode, steps, step0 and the mode's
// own fields set and all else zero; the caller has checked its own arguments.
int launch_step(vlg::StepParams& p, const void* packed, int K, int X, int K_active, int N, int T, int n_poly, int M,
                const float* a, const float* b, const float* omega, const float* basis, const float* t,
                const uint8_t* draws, const int32_t* decoder_base, uint64_t seed, int64_t curve_id0, int precision,
                void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_device();
  if (rc != VLG_OK) return rc;
  if (!packed || N <= 0 || T < 2 || n_poly < 1 || M < 1 || K_active < 1) return VLG_ERR_INVALID_ARGUMENT;
  // MC samples: the fp32 kernel holds all of them at once (<= MAX_M); the tensor-core kernel walks blocks of two (<= 64)
  if (n_poly > vlg::MAX_NPOLY || M > (precision == VLG_PRECISION_FP32 ? vlg::MAX_M : 64) || K_active > 254) return VLG_ERR_UNSUPPORTED;
  if (precision < VLG_PRECISION_FP32 || precision > VLG_PRECISION_F16X3F) return VLG_ERR_INVALID_ARGUMENT;
  if (vlg_packed_decoders_bytes(K, vlg::H, X) == 0 || K_active > K) return VLG_ERR_INVALID_ARGUMENT;
  if (workspace_bytes < vlg_workspace_bytes(N, T, n_poly, K_active, M, precision)) return VLG_ERR_WORKSPACE;
  p.packed = packed;
  p.K = K_active;
  p.K_total = K;
  p.X = X;
  p.N = N;
  p.T = T;
  p.n_poly = n_poly;
  p.Kb = n_poly + 1;
  p.M = M;
  p.a = a;
  p.b = b;
  p.omega = const_cast<float*>(omega);   // written only by StepMode::Optimize
  p.basis = basis;
  p.t = t;
  p.draws = draws;
  p.dec_base = decoder_base;
  p.seed = seed;
  p.curve_id0 = curve_id0;
  p.workspace = workspace;
  p.workspace_bytes = workspace_bytes;
  p.precision = precision;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const cudaError_t e = precision == VLG_PRECISION_FP32 ? vlg::launch_simt(p, st) : vlg::launch_tc(p, st);
  if (e == cudaErrorNotSupported) return VLG_ERR_UNSUPPORTED;
  return e == cudaSuccess ? VLG_OK : cuda_fail(e);
}

}  // namespace

extern "C" {

const char* vlg_error_string(int code) {
  switch (code) {
    case VLG_OK: return "ok";
    case VLG_ERR_INVALID_ARGUMENT: return "invalid argument";
    case VLG_ERR_UNSUPPORTED: return "unsupported shape or option";
    case VLG_ERR_CUDA: return "CUDA error (see vlg_last_cuda_error)";
    case VLG_ERR_DEVICE: return "current device is not an sm_100 (B200) GPU";
    case VLG_ERR_WORKSPACE: return "workspace too small";
    case VLG_ERR_NUMERIC: return "non-finite energy/omega (fp16 operand overflow?) or out-of-range draw in the last launch";
    default: return "unknown error";
  }
}

const char* vlg_last_cuda_error(void) { return g_cuda_err; }

int vlg_abi_version(void) { return VLG_ABI_VERSION; }

size_t vlg_packed_decoders_bytes(int K, int H, int X) {
  // X is limited by the Diff row stride of the kernels (52 floats)
  if (K < 1 || K > 254 || H != vlg::H || X < 1 || X > 52) return 0;
  return sizeof(vlg::PackedHeader) + size_t(K) * vlg::DEC_FLOATS * sizeof(float);
}

int vlg_pack_decoders(const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                      const float* b3, int K, int H, int X, void* packed, void* stream) {
  if (!W1 || !b1 || !W2 || !b2 || !W3 || !b3 || !packed) return VLG_ERR_INVALID_ARGUMENT;
  if (vlg_packed_decoders_bytes(K, H, X) == 0) return VLG_ERR_UNSUPPORTED;
  int rc = check_device();
  if (rc != VLG_OK) return rc;
  cudaError_t e = vlg::launch_pack(W1, b1, W2, b2, W3, b3, K, X, packed, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? VLG_OK : cuda_fail(e);
}

size_t vlg_workspace_bytes(int N, int T, int n_poly, int K_active, int M, int precision) {
  (void)n_poly;
  if (precision == VLG_PRECISION_FP32) return vlg::simt_workspace_bytes(N, T, K_active, M);
  return vlg::tc_workspace_bytes(N, T, K_active, M);
}

int vlg_optimize_steps(const void* packed, int K, int X, int K_active, int N, int T, int n_poly, int M, int steps, int step0,
                       const float* a, const float* b, float* omega, float* adam_m, float* adam_v,
                       const float* basis, const float* t, const uint8_t* draws, const int32_t* decoder_base, uint64_t seed,
                       int64_t curve_id0, double lr, double beta1, double beta2, double eps, double penalty_w, float* energy_last,
                       float* energy_trace, int precision, void* workspace, size_t workspace_bytes, void* stream) {
  if (!a || !b || !omega || !adam_m || !adam_v || !basis || !t || steps < 0 || step0 < 0)
    return VLG_ERR_INVALID_ARGUMENT;
  if (steps == 0) return VLG_OK;
  vlg::StepParams p{};
  p.mode = vlg::StepMode::Optimize;
  p.steps = steps;
  p.step0 = step0;
  p.adam_m = adam_m;
  p.adam_v = adam_v;
  p.lr = lr;
  p.beta1 = beta1;
  p.beta2 = beta2;
  p.eps = float(eps);
  p.one_minus_b1 = float(1.0 - beta1);
  p.beta2f = float(beta2);
  p.one_minus_b2 = float(1.0 - beta2);
  p.penalty_w = float(penalty_w);
  p.energy_last = energy_last;
  p.energy_trace = energy_trace;
  return launch_step(p, packed, K, X, K_active, N, T, n_poly, M, a, b, omega, basis, t, draws, decoder_base, seed,
                     curve_id0, precision, workspace, workspace_bytes, stream);
}

int vlg_workspace_status(const void* workspace, int* flags, void* stream) {
  if (!workspace) return VLG_ERR_INVALID_ARGUMENT;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned int word = 0;
  // word [1] of the workspace header of both step kernels (zeroed by their launchers)
  cudaError_t e = cudaMemcpyAsync(&word, static_cast<const unsigned int*>(workspace) + 1, sizeof(word),
                                  cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return cuda_fail(e);
  if (flags) *flags = int(word);
  return word == 0 ? VLG_OK : VLG_ERR_NUMERIC;
}

int vlg_workspace_counters(const void* workspace, unsigned long long* counters, void* stream) {
  if (!workspace || !counters) return VLG_ERR_INVALID_ARGUMENT;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaError_t e = cudaMemcpyAsync(counters, static_cast<const unsigned int*>(workspace) + 2,
                                  2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  return e == cudaSuccess ? VLG_OK : cuda_fail(e);
}

int vlg_curve_energy(const void* packed, int K, int X, int K_active, int N, int T, int n_poly, int M, const float* a,
                     const float* b, const float* omega, const float* basis, const float* t, const uint8_t* draws,
                     const int32_t* decoder_base, uint64_t seed, int64_t curve_id0, int step, float* energy, float* length, int precision,
                     void* workspace, size_t workspace_bytes, void* stream) {
  if (!a || !b || !omega || !basis || !t || !energy || step < 0) return VLG_ERR_INVALID_ARGUMENT;
  vlg::StepParams p{};
  p.mode = vlg::StepMode::Energy;
  p.steps = 1;
  p.step0 = step;
  p.energy_last = energy;
  p.length_out = length;
  return launch_step(p, packed, K, X, K_active, N, T, n_poly, M, a, b, omega, basis, t, draws, decoder_base, seed,
                     curve_id0, precision, workspace, workspace_bytes, stream);
}

int vlg_curve_energy_grad(const void* packed, int K, int X, int K_active, int N, int T, int n_poly, int M,
                          const float* a, const float* b, const float* omega, const float* basis, const float* t,
                          const uint8_t* draws, const int32_t* decoder_base, uint64_t seed, int64_t curve_id0, int step,
                          float* energy, float* grad_omega, float* grad_a, float* grad_b, int precision,
                          void* workspace, size_t workspace_bytes, void* stream) {
  if (!a || !b || !omega || !basis || !t || !energy || !grad_omega || !grad_a || !grad_b || step < 0)
    return VLG_ERR_INVALID_ARGUMENT;
  // one step of the optimiser's kernel in gradient-output mode: same draw stream as vlg_curve_energy at `step`
  vlg::StepParams p{};
  p.mode = vlg::StepMode::EnergyGrad;
  p.steps = 1;
  p.step0 = step;
  p.energy_last = energy;
  p.grad_omega = grad_omega;
  p.grad_a = grad_a;
  p.grad_b = grad_b;
  return launch_step(p, packed, K, X, K_active, N, T, n_poly, M, a, b, omega, basis, t, draws, decoder_base, seed,
                     curve_id0, precision, workspace, workspace_bytes, stream);
}

int vlg_ensemble_std_norm(const void* packed, int K, int X, int K_active, int G, const float* grid, float* out,
                          void* stream) {
  if (!packed || !grid || !out || G <= 0 || K_active < 1) return VLG_ERR_INVALID_ARGUMENT;
  if (vlg_packed_decoders_bytes(K, vlg::H, X) == 0 || K_active > K) return VLG_ERR_INVALID_ARGUMENT;
  int rc = check_device();
  if (rc != VLG_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaError_t e = vlg::launch_std_norm(packed, K_active, X, G, grid, out, st);
  return e == cudaSuccess ? VLG_OK : cuda_fail(e);
}

}  // extern "C"

namespace {

// What vlg_decode and vlg_decode_backward share: argument checks (before any CUDA call), the device check, the launch.
int decode_entry(const void* packed, int K, int X, int K_active, int P, const float* z, const float* dx, float* x, float* dz,
                 int precision, void* workspace, size_t workspace_bytes, void* stream) {
  if (!packed || !z || !(x || dz) || (dz && !dx) || !workspace || P <= 0 || K_active < 1 || K_active > K)
    return VLG_ERR_INVALID_ARGUMENT;
  if (precision < VLG_PRECISION_FP32 || precision > VLG_PRECISION_F16X3F) return VLG_ERR_INVALID_ARGUMENT;
  if (vlg_packed_decoders_bytes(K, vlg::H, X) == 0) return VLG_ERR_INVALID_ARGUMENT;
  if (precision != VLG_PRECISION_FP32 && K_active > 128) return VLG_ERR_UNSUPPORTED;
  if (workspace_bytes < VLG_DECODE_WORKSPACE_BYTES) return VLG_ERR_WORKSPACE;
  int rc = check_device();
  if (rc != VLG_OK) return rc;
  cudaError_t e = vlg::launch_decode(packed, K, X, K_active, P, z, dx, x, dz, precision, workspace,
                                     static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? VLG_OK : cuda_fail(e);
}

}  // namespace

extern "C" {

int vlg_decode(const void* packed, int K, int X, int K_active, int P, const float* z, float* x, int precision,
               void* workspace, size_t workspace_bytes, void* stream) {
  if (!x) return VLG_ERR_INVALID_ARGUMENT;
  return decode_entry(packed, K, X, K_active, P, z, nullptr, x, nullptr, precision, workspace, workspace_bytes, stream);
}

int vlg_decode_backward(const void* packed, int K, int X, int K_active, int P, const float* z, const float* dx,
                        float* dz, int precision, void* workspace, size_t workspace_bytes, void* stream) {
  if (!dx || !dz) return VLG_ERR_INVALID_ARGUMENT;
  return decode_entry(packed, K, X, K_active, P, z, dx, nullptr, dz, precision, workspace, workspace_bytes, stream);
}

size_t vlg_expected_energy_workspace_bytes(int N, int T, int X) {
  if (N < 1 || T < 2 || X < 1 || X > 52 || size_t(T) * size_t(N) > size_t(INT_MAX)) return 0;
  const size_t P = size_t(T) * size_t(N);
  return VLG_DECODE_WORKSPACE_BYTES + (P * size_t(X) + P) * sizeof(float);
}

int vlg_expected_energy(const void* packed, int K, int X, int K_active, int N, int T, const float* z, float* energy,
                        float* grad_z, int precision, void* workspace, size_t workspace_bytes, void* stream) {
  if (!packed || !z || !energy || !workspace || N < 1 || T < 2 || K_active < 1 || K_active > K)
    return VLG_ERR_INVALID_ARGUMENT;
  if (size_t(T) * size_t(N) > size_t(INT_MAX)) return VLG_ERR_INVALID_ARGUMENT;
  if (precision < VLG_PRECISION_FP32 || precision > VLG_PRECISION_F16X3F) return VLG_ERR_INVALID_ARGUMENT;
  if (vlg_packed_decoders_bytes(K, vlg::H, X) == 0) return VLG_ERR_INVALID_ARGUMENT;
  if (precision != VLG_PRECISION_FP32 && K_active > 128) return VLG_ERR_UNSUPPORTED;
  if (workspace_bytes < vlg_expected_energy_workspace_bytes(N, T, X)) return VLG_ERR_WORKSPACE;
  int rc = check_device();
  if (rc != VLG_OK) return rc;
  cudaError_t e = vlg::launch_expected_energy(packed, K, X, K_active, N, T, z, energy, grad_z, precision, workspace,
                                              static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? VLG_OK : cuda_fail(e);
}

int vlg_spline_points(int N, int T, int n_poly, const float* a, const float* b, const float* omega,
                      const float* basis, const float* t, float* z, void* stream) {
  if (!a || !b || !omega || !basis || !t || !z || N <= 0 || T <= 0 || n_poly < 1) return VLG_ERR_INVALID_ARGUMENT;
  if (n_poly > vlg::MAX_NPOLY) return VLG_ERR_UNSUPPORTED;
  int rc = check_device();
  if (rc != VLG_OK) return rc;
  cudaError_t e = vlg::launch_spline_points(N, T, n_poly, a, b, omega, basis, t, z, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? VLG_OK : cuda_fail(e);
}

int vlg_spline_points_backward(int N, int T, int n_poly, const float* basis, const float* t, const float* dz,
                               float* grad_omega, float* grad_a, float* grad_b, void* stream) {
  if (!basis || !t || !dz || !grad_omega || !grad_a || !grad_b || N <= 0 || T <= 0 || n_poly < 1)
    return VLG_ERR_INVALID_ARGUMENT;
  if (n_poly > vlg::MAX_NPOLY) return VLG_ERR_UNSUPPORTED;
  int rc = check_device();
  if (rc != VLG_OK) return rc;
  cudaError_t e = vlg::launch_spline_points_backward(N, T, n_poly, basis, t, dz, grad_omega, grad_a, grad_b,
                                                     static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? VLG_OK : cuda_fail(e);
}

int vlg_fit_splines(int N, int Lmax, int n_poly, const float* targets, const int32_t* lens, const float* basis,
                    float* omega, float* ab, void* stream) {
  if (!targets || !lens || !basis || !omega || !ab || N <= 0 || Lmax < 2 || n_poly < 1)
    return VLG_ERR_INVALID_ARGUMENT;
  if (n_poly > vlg::MAX_NPOLY) return VLG_ERR_UNSUPPORTED;
  int rc = check_device();
  if (rc != VLG_OK) return rc;
  cudaError_t e =
      vlg::launch_fit_splines(N, Lmax, n_poly, targets, lens, basis, omega, ab, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? VLG_OK : cuda_fail(e);
}

}  // extern "C"
