// Internal launch interface between the C-ABI front end (vlg_api.cu) and the kernels.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <type_traits>

#include "../../include/vlg.h"

namespace vlg {

// What a step-kernel launch computes:
//   Optimize   (vlg_optimize_steps)    `steps` Adam steps; writes omega, adam_m, adam_v and the energies back
//   Energy     (vlg_curve_energy)      the energy (and poly-line length) of one step, no backward items
//   EnergyGrad (vlg_curve_energy_grad) the energy of one step and dE/d(omega), dE/da, dE/db of the energy alone
//                                      (no penalty term); no Adam, omega is read only
enum class StepMode { Optimize, Energy, EnergyGrad };

// Calls f(std::integral_constant<StepMode, m>{}) for the launch's mode m: the kernels take the mode as a template
// parameter, so that no mode carries the code of another.
template <class F>
auto with_mode(StepMode m, F&& f) {
  switch (m) {
    case StepMode::Energy: return f(std::integral_constant<StepMode, StepMode::Energy>{});
    case StepMode::EnergyGrad: return f(std::integral_constant<StepMode, StepMode::EnergyGrad>{});
    default: return f(std::integral_constant<StepMode, StepMode::Optimize>{});
  }
}

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
  float* adam_m;               // Optimize only
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
  float* length_out;           // [N] or null (Energy only)
  float* grad_omega;           // [N,Kb,2] (EnergyGrad only)
  float* grad_a;               // [N,2]    (EnergyGrad only)
  float* grad_b;               // [N,2]    (EnergyGrad only)
  void* workspace;
  size_t workspace_bytes;
  int precision;
  StepMode mode;
};

// Launch planning shared by both step kernels (vlg_api.cu).
// CTAs of a persistent launch over N work units: one per SM, at most N.
int persistent_grid(int N);
// Expected 128-row items of one decoder in a window of w points, each of which draws the decoder with probability p:
// its row count n is ~Binomial(w, p) (normal approximation) and it costs ceil(n / 128) items.
double expected_items(int w, double p);

size_t simt_workspace_bytes(int N, int T, int K, int M);
cudaError_t launch_simt(const StepParams& p, cudaStream_t stream);

size_t tc_workspace_bytes(int N, int T, int K, int M);
cudaError_t launch_tc(const StepParams& p, cudaStream_t stream);

cudaError_t launch_pack(const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                        const float* b3, int K, int X, void* packed, cudaStream_t stream);
cudaError_t launch_std_norm(const void* packed, int K, int X, int G, const float* grid, float* out,
                            cudaStream_t stream);
cudaError_t launch_spline_points(int N, int T, int n_poly, const float* a, const float* b, const float* omega,
                                 const float* basis, const float* t, float* z, cudaStream_t stream);
cudaError_t launch_spline_points_backward(int N, int T, int n_poly, const float* basis, const float* t, const float* dz,
                                          float* grad_omega, float* grad_a, float* grad_b, cudaStream_t stream);
// Decoder ensemble outputs (dz == nullptr) or their input gradient (x unused); vlg_decode.cu
cudaError_t launch_decode(const void* packed, int K_total, int X, int K, int P, const float* z, const float* dx, float* x,
                          float* dz, int precision, void* workspace, cudaStream_t stream);
// Expected ensemble curve energy of the curves z [T][N][2] and, if grad_z is not null, dE_n/dz; vlg_decode.cu.
// workspace: the 256-byte status header, then mu [T*N*X] and e [T*N] floats (vlg_expected_energy_workspace_bytes)
cudaError_t launch_expected_energy(const void* packed, int K_total, int X, int K, int N, int T, const float* z,
                                   float* energy, float* grad_z, int precision, void* workspace, cudaStream_t stream);
cudaError_t launch_fit_splines(int N, int Lmax, int n_poly, const float* targets, const int32_t* lens,
                               const float* basis, float* omega, float* ab, cudaStream_t stream);

}  // namespace vlg
