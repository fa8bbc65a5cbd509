// Internal launch interface between the C-ABI front end (vlg_api.cu) and the kernels.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/vlg.h"

namespace vlg {

struct StepParams {
  const void* packed;
  int K, X;                    // active decoders, output width
  int K_total;                 // decoders in `packed`
  int N, T, n_poly, Kb, M;
  int steps, step0;
  int unit_steps;              // Adam steps per work unit (set by the tensor-core launcher)
  const float* a;
  const float* b;
  float* omega;
  float* adam_m;
  float* adam_v;
  const float* basis;
  const float* t;
  const uint8_t* draws;        // [N][steps][M][2][T-1] or null
  const int32_t* dec_base;     // [N] or null: curve n uses decoders dec_base[n] .. dec_base[n] + K - 1 of `packed`
  uint64_t seed;
  int64_t curve_id0;
  double lr, beta1, beta2;
  float eps, one_minus_b1, beta2f, one_minus_b2, penalty_w;
  float* energy_last;          // [N] or null
  float* energy_trace;         // [steps][N] or null
  float* length_out;           // [N] or null (forward-only mode)
  // gradient-output mode (vlg_curve_energy_grad; null otherwise): the GRAD kernels write dE/d(omega), dE/da and
  // dE/db of the energy alone (no penalty term) and skip Adam; omega is read only, adam_m / adam_v are null
  float* grad_omega;           // [N,Kb,2]
  float* grad_a;               // [N,2]
  float* grad_b;               // [N,2]
  void* workspace;
  size_t workspace_bytes;
  int precision;
};

size_t simt_smem_bytes(int T, int K, int M);
size_t simt_workspace_bytes(int N, int T, int K, int M);
cudaError_t launch_simt(const StepParams& p, bool grad, cudaStream_t stream);

size_t tc_workspace_bytes(int N, int T, int K, int M);
cudaError_t launch_tc(const StepParams& p, bool grad, cudaStream_t stream);

cudaError_t launch_pack(const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                        const float* b3, int K, int X, void* packed, cudaStream_t stream);
cudaError_t launch_std_norm(const void* packed, int K, int X, int G, const float* grid, float* out,
                            cudaStream_t stream);
cudaError_t launch_spline_points(int N, int T, int n_poly, const float* a, const float* b, const float* omega,
                                 const float* basis, const float* t, float* z, cudaStream_t stream);
cudaError_t launch_spline_points_backward(int N, int T, int n_poly, const float* basis, const float* t, const float* dz,
                                          float* grad_omega, float* grad_a, float* grad_b, cudaStream_t stream);
cudaError_t launch_fit_splines(int N, int Lmax, int n_poly, const float* targets, const int32_t* lens,
                               const float* basis, float* omega, float* ab, cudaStream_t stream);

}  // namespace vlg
