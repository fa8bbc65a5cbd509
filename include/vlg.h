/*
 * vlg.h -- C ABI of the B200-native geodesic curve-energy engine (libvlg_b200.so).
 *
 * The reference (johannefranck/vae-latent-geometry) is pure Python/PyTorch and has no FFI
 * of its own; the seam this library sits behind is the Python inner loop
 *     src/optimize.py:155-162   (ensemble optimisation, the headline path)
 *     src/eval.py:119-125       (CoV study, decoders[:k])
 *     src/single_decoder/optimize_energy_batched.py:95-102 (single decoder)
 * plus the forward-only evaluations listed per entry point below.  INTEGRATION.md shows
 * the ctypes / torch.library binding a maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer on the current CUDA device unless stated;
 *     the caller owns every buffer; nothing is allocated, nothing is synchronised
 *     (vlg_workspace_status is the one documented exception): work is enqueued on
 *     `stream` (a cudaStream_t passed as void*).  The library keeps no per-buffer state:
 *     the caller passes the packed ensemble's K and X with every call.
 *   - all arrays are dense, row-major, fp32 unless stated.
 *   - every function returns 0 on success or a negative VLG_ERR_* code; it never throws.
 *   - requires an sm_100 (B200) device: there is no CPU or other-arch fallback.
 *
 * Shapes (names follow the reference): N curves, T points per curve (t grid), n_poly
 * cubic segments, Kb = n_poly+1 free coefficients per latent dim, K decoders
 * 2 -> H(=128) -> H -> X (1 <= X <= 52; 50 for tasic-pca50), M Monte-Carlo decoder pairings.
 * Limits (VLG_ERR_UNSUPPORTED beyond them): n_poly <= 8; K_active <= 254 with VLG_PRECISION_FP32, <= 128 on the
 * tensor-core precisions; M <= 4 with VLG_PRECISION_FP32, <= 64 on the tensor-core precisions (blocks of two).
 */
#ifndef VLG_H_
#define VLG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VLG_ABI_VERSION 2

enum {
  VLG_OK = 0,
  VLG_ERR_INVALID_ARGUMENT = -1, /* null pointer, non-positive size, ...              */
  VLG_ERR_UNSUPPORTED = -2,      /* shape outside what the kernels are built for      */
  VLG_ERR_CUDA = -3,             /* a CUDA runtime call failed (see vlg_last_cuda_error) */
  VLG_ERR_DEVICE = -4,           /* current device is not sm_100                      */
  VLG_ERR_WORKSPACE = -5,        /* workspace too small                               */
  VLG_ERR_NUMERIC = -6           /* vlg_workspace_status: the last launch saw a non-finite energy / omega
                                    (fp16 operand overflow) or an out-of-range explicit draw          */
};

/* Status flags a step kernel leaves in its workspace (read back by vlg_workspace_status). */
enum {
  VLG_STATUS_BAD_DRAW = 1,  /* an explicit draw was >= K_active (the kernel clamped it to K_active-1) */
  VLG_STATUS_BAD_PACKED = 4, /* `packed` does not start with a header of the K / X the caller passed */
  VLG_STATUS_NONFINITE = 2  /* an energy, an updated omega or (vlg_curve_energy_grad) a gradient component was
                               inf/NaN: with VLG_PRECISION_F16* this is what an operand beyond the fp16 range
                               (65504) turns into                                                      */
};

/* Arithmetic used for the two 128-wide decoder layers (and their transposes). */
enum {
  VLG_PRECISION_FP32 = 0,   /* CUDA-core FFMA, fp32 accumulate: the <=1e-4/step variant     */
  VLG_PRECISION_TF32 = 1,   /* tcgen05.mma kind::tf32, fp32 accumulate in TMEM              */
  VLG_PRECISION_F16X3 = 2,  /* 3-term split on the tensor pipe: operands as hi + lo fp16 pairs (~21 bits),
                               hi*hi + lo*hi + hi*lo in the fp32 accumulator: fp32-grade (measured 2e-6
                               relative per-step energy), 5-6x the speed of the CUDA-core kernel       */
  VLG_PRECISION_TF32X3 = 2, /* former name of the same slot */
  VLG_PRECISION_F16 = 3,    /* tcgen05.mma kind::f16: fp16 operands (11-bit significand, as TF32; backward
                               quantities pre-scaled by 2^6), fp32 accumulate in TMEM: half the tensor-pipe
                               time and weight traffic of TF32 for the same <=1e-3 length tolerance     */
  VLG_PRECISION_F16X3F = 4  /* 3-term split in the forward GEMMs (energies and lengths fp32-grade, as F16X3),
                               single-term fp16 operands in the backward GEMMs (gradient to ~2.5e-4 relative) */
};

const char* vlg_error_string(int code);
/* Text of the last CUDA error seen by this library on the calling thread ("" if none). */
const char* vlg_last_cuda_error(void);
int vlg_abi_version(void);

/* ---- decoder weights -------------------------------------------------------------
 * Replaces `decoders = list(model.decoder)` (src/optimize.py:103): one-time repack of
 * the K decoder MLPs (src/train.py:80-85; single VAE: src/single_decoder/vae.py:29-42
 * with only the first X rows of the last layer) into the kernels' layouts.
 *   W1[K,H,2] b1[K,H] W2[K,H,H] b2[K,H] W3[K,X,H] b3[K,X]   (nn.Linear weight layout)
 *   packed: device buffer of vlg_packed_decoders_bytes(K,H,X) bytes, 256-byte aligned.
 */
size_t vlg_packed_decoders_bytes(int K, int H, int X);
int vlg_pack_decoders(const float* W1, const float* b1, const float* W2, const float* b2,
                      const float* W3, const float* b3, int K, int H, int X, void* packed,
                      void* stream);

/* Scratch the optimiser needs (0 is a valid answer). */
size_t vlg_workspace_bytes(int N, int T, int n_poly, int K_active, int M, int precision);

/* ---- the hot loop ------------------------------------------------------------------
 * Replaces src/optimize.py:155-162 (and its twins) for `steps` Adam steps of all N
 * curves: spline evaluation (src/optimize.py:22-35), all-decoder forward
 * (src/train.py:42-46), MC pair energy (src/optimize.py:38-75), end-point penalty
 * (158-160), backward to omega (161; decoder weight gradients are not formed), Adam
 * (162; torch defaults, bias correction uses step0+s+1).
 *
 *   packed      from vlg_pack_decoders (of K decoders with X outputs: the caller passes the same
 *               K and X it packed with); the first K_active decoders are used
 *               (`model.decoder[:k]`, src/eval.py:113)
 *   a, b        [N,2]      end points
 *   omega       [N,Kb,2]   in: current coefficients; out: after `steps` updates
 *   adam_m/v    [N,Kb,2]   in/out Adam moments (zeros for a fresh optimiser)
 *   basis       [4*n_poly,Kb]  from the spline file (never recomputed, SURVEY hard part 7)
 *   t           [T]        the grid torch.linspace(0,1,T) (src/optimize.py:130)
 *   draws       NULL, or uint8 [N,steps,M,2,T-1]: explicit decoder indices < K_active
 *               (role 0 = d1 at point t, role 1 = d2 at point t+1; src/optimize.py:57-61);
 *               a value >= K_active is clamped and flagged (VLG_STATUS_BAD_DRAW).
 *               NULL -> counter-based Philox4x32-10 stream keyed on
 *               (seed, curve_id0+n, step0+s, m, t): independent of sharding.
 *   decoder_base NULL, or int32 [N]: curve n uses decoders decoder_base[n] .. decoder_base[n]+K_active-1 of
 *               `packed` instead of 0 .. K_active-1 -- several weight sets (the ensembles of several training
 *               seeds, src/eval.py:94-113) packed into one buffer and optimised in ONE launch; draws stay
 *               relative to the curve's own set.  Out-of-range bases are flagged (VLG_STATUS_BAD_PACKED).
 *   energy_last [N]        energy evaluated in the LAST step (before its update), i.e.
 *               what src/optimize.py:168 turns into geodesic_length = sqrt(energy)
 *   energy_trace NULL or [steps,N]: energy of every step (src/optimize.py:164-165)
 *   lr..penalty_w are doubles because torch keeps them as Python floats and rounds the
 *   derived scalars (1-beta1, lr/(1-beta1^s), ...) to fp32 only when applying them.
 */
int vlg_optimize_steps(const void* packed, int K, int X, int K_active, int N, int T, int n_poly, int M,
                       int steps, int step0, const float* a, const float* b, float* omega,
                       float* adam_m, float* adam_v, const float* basis, const float* t,
                       const uint8_t* draws, const int32_t* decoder_base, uint64_t seed, int64_t curve_id0, double lr,
                       double beta1, double beta2, double eps, double penalty_w,
                       float* energy_last, float* energy_trace, int precision,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Status of the last vlg_optimize_steps / vlg_curve_energy / vlg_curve_energy_grad / vlg_decode* /
 * vlg_expected_energy launch that used `workspace` (the word sits at the same place in every one): copies the
 * status word back and SYNCHRONISES `stream` (the only entry point that does).  *flags (host
 * pointer, may be NULL) receives the VLG_STATUS_* bits; returns VLG_OK when none is set, else
 * VLG_ERR_NUMERIC.  Replaces the finite-check a caller of the reference would do on `energy`
 * (the reference itself never checks: src/optimize.py:164-168 prints whatever it gets). */
int vlg_workspace_status(const void* workspace, int* flags, void* stream);

/* Work statistics of the last tensor-core launch that used `workspace` (SYNCHRONISES `stream`):
 * counters[0] = 128-row decoder items executed (each = the four tcgen05 GEMMs of one decoder on up to 128
 * selected curve points; forward-only launches run two of them), counters[1] = occupied rows of those items.
 * Row compaction makes the executed tensor FLOPs smaller than the algorithmic K x T count (DESIGN.md §4);
 * bench.py reports both.  counters is a HOST pointer to two uint64.  Zero for the fp32 kernel. */
int vlg_workspace_counters(const void* workspace, unsigned long long* counters, void* stream);

/* ---- forward-only evaluation --------------------------------------------------------
 * energy[N]  = compute_energy_mc (src/optimize.py:38-75) for the given omega and draws
 *              (draws: uint8 [N,1,M,2,T-1] or NULL -> counter stream at step `step`).
 *              With K_active=1, M=1 this is the deterministic single-decoder energy
 *              (src/single_decoder/optimize_energy_batched.py:51-57).
 * length[N]  = (1/M) sum_m sum_t ||x2 - x1||  (NULL to skip); with K_active=1, M=1 it is
 *              compute_geodesic_lengths (optimize_energy_batched.py:42-49).
 * The ensemble "geodesic_length" of src/optimize.py:168 / src/eval.py:127 is sqrt(energy).
 */
int vlg_curve_energy(const void* packed, int K, int X, int K_active, int N, int T, int n_poly, int M,
                     const float* a, const float* b, const float* omega, const float* basis,
                     const float* t, const uint8_t* draws, const int32_t* decoder_base, uint64_t seed, int64_t curve_id0,
                     int step, float* energy, float* length, int precision, void* workspace,
                     size_t workspace_bytes, void* stream);

/* ---- differentiable energy --------------------------------------------------------------
 * Replaces the autograd backward of the energy at src/optimize.py:161 (`loss.sum().backward()`, the energy's
 * part of it): ONE launch of the optimiser's step kernel that evaluates energy[N] exactly as vlg_curve_energy
 * (same arguments, same draw stream at `step`) and its gradient with respect to the curve parameters
 *   grad_omega [N,Kb,2] = dE/d(omega) = sum_t P[t]^T dz[t]
 *   grad_a     [N,2]    = dE/da      = sum_t (1-t) dz[t]
 *   grad_b     [N,2]    = dE/db      = sum_t t dz[t]
 * where dz[t] = dE/dz[t] flows back through the decoders (decoder weight gradients are not formed).  The energy
 * alone: no end-point penalty term (the reference's compute_energy_mc has none), no Adam, omega is not written.
 * The energy is bit-identical to the first step of vlg_optimize_steps with the same inputs; grad_omega is the
 * gradient that step hands to Adam minus its penalty term.  All output pointers are required; the workspace is
 * vlg_workspace_bytes as for the other step-kernel calls and vlg_workspace_status reads its status.
 */
int vlg_curve_energy_grad(const void* packed, int K, int X, int K_active, int N, int T, int n_poly, int M,
                          const float* a, const float* b, const float* omega, const float* basis,
                          const float* t, const uint8_t* draws, const int32_t* decoder_base, uint64_t seed,
                          int64_t curve_id0, int step, float* energy, float* grad_omega, float* grad_a,
                          float* grad_b, int precision, void* workspace, size_t workspace_bytes, void* stream);

/* ---- ensemble disagreement field ------------------------------------------------------
 * out[g] = || std_k f_k(grid[g]) ||_2 over the first K_active decoders, unbiased std
 * (src/init_splines_ensemble.py:49-51, before the min-max normalisation).  grid [G,2].
 */
int vlg_ensemble_std_norm(const void* packed, int K, int X, int K_active, int G, const float* grid,
                          float* out, void* stream);

/* ---- decoder ensemble outputs and their input gradient ----------------------------------------
 * x[k,p,:] = f_k(z[p]) for the first K_active decoders of `packed`: the reference's
 *   torch.stack([d(z).mean for d in decoders])   (src/optimize.py:50, src/init_splines_ensemble.py:49,
 *                                                 the decoder check at src/optimize.py:108-116)
 * with f_k the 2 -> 128 -> ReLU -> 128 -> ReLU -> X MLP of src/train.py:80-85.  z [P,2], x [K_active,P,X], fp32,
 * contiguous; offsets are 64-bit (K_active * P * X may exceed 2^31).
 * vlg_decode_backward: dz[p] = sum_k W1^T (m1 . W2^T (m2 . W3^T dx[k,p])), the input gradient autograd forms for a
 * loss on those outputs (no weight gradients).  dx [K_active,P,X], dz [P,2].  The ReLU masks m1, m2 are recomputed
 * from z, so the two calls share no state.  The decoders are summed in a fixed order with no atomics: repeated calls
 * give the same bits, and each point's dz does not depend on the other points.  Each row of dx is normalised by a power
 * of two before it is rounded to a tensor-core operand, so the result scales exactly with dx.
 * Precision: any VLG_PRECISION_*; the tensor-core ones need K_active <= 128 (VLG_ERR_UNSUPPORTED beyond).
 * VLG_PRECISION_F16X3F runs the forward GEMMs as F16X3 and the backward GEMMs (B3, B2) single-term.
 * workspace: VLG_DECODE_WORKSPACE_BYTES; vlg_workspace_status reads the launch's status (VLG_STATUS_BAD_PACKED,
 * VLG_STATUS_NONFINITE for a non-finite z, x or dz component).  Asynchronous on `stream`; allocates nothing.
 * Argument errors are returned before any CUDA call.
 */
#define VLG_DECODE_WORKSPACE_BYTES 256   /* status header read by vlg_workspace_status */
int vlg_decode(const void* packed, int K, int X, int K_active, int P, const float* z, float* x,
               int precision, void* workspace, size_t workspace_bytes, void* stream);
int vlg_decode_backward(const void* packed, int K, int X, int K_active, int P, const float* z, const float* dx,
                        float* dz, int precision, void* workspace, size_t workspace_bytes, void* stream);

/* ---- expected ensemble curve energy ------------------------------------------------------------
 * The M -> infinity limit of compute_energy_mc (src/optimize.py:38-75) for curves given as points z [T][N][2] (a
 * spline's model(t_vals), a Dijkstra poly-line, ...): with x_k(t) = f_k(z_t) for the first K_active decoders,
 *   energy[n] = sum_{t<T-1} E_{k,l} ||f_l(z_{t+1}) - f_k(z_t)||^2 = sum_t ||mu_{t+1} - mu_t||^2 + sum_t c_t V_t
 *   mu_t = (1/K) sum_k x_k(t),  V_t = (1/K) sum_k ||x_k(t) - mu_t||^2,  c_t = 1 at the two ends, 2 inside,
 * and, when grad_z is not NULL, grad_z[t][n] = dE_n/dz_t = (2/K) sum_k J_k(z_t)^T (c_t x_k(t) - mu_{t-1} - mu_{t+1})
 * (only the neighbours that exist).  Three passes: every decoder's forward for the means, every decoder's forward
 * again (and the backward for grad_z) for V_t and each point's energy term, and a fixed-order sum over t per curve.
 * No atomics: repeated calls give the same bits, and a curve's energy and grad_z do not depend on the other curves.
 * N >= 1, T >= 2, T * N <= INT_MAX; precision and the K_active / X limits as for vlg_decode; VLG_PRECISION_F16X3F
 * runs the forward GEMMs 3-term and the backward GEMMs single-term.  workspace: at least
 * vlg_expected_energy_workspace_bytes(N, T, X) bytes (the 256-byte status header, then mu [T*N*X] and the energy
 * terms [T*N] floats; 0 for a shape outside the limits); vlg_workspace_status reads the launch's status
 * (VLG_STATUS_BAD_PACKED, VLG_STATUS_NONFINITE for a non-finite z, mean, energy term, energy or grad_z component).
 * Asynchronous on `stream`; allocates nothing.  Argument errors are returned before any CUDA call.
 */
size_t vlg_expected_energy_workspace_bytes(int N, int T, int X);
int vlg_expected_energy(const void* packed, int K, int X, int K_active, int N, int T, const float* z, float* energy,
                        float* grad_z, int precision, void* workspace, size_t workspace_bytes, void* stream);

/* ---- spline evaluation ----------------------------------------------------------------
 * z[T,N,2] = GeodesicSplineBatch.forward(t) (src/optimize.py:22-35).  Used by the drop-in
 * writers / plotting helpers; also handy for testing.
 */
int vlg_spline_points(int N, int T, int n_poly, const float* a, const float* b,
                      const float* omega, const float* basis, const float* t, float* z,
                      void* stream);

/* Backward of vlg_spline_points: the spline's part of the autograd backward at src/optimize.py:161 (the
 * end-point penalty `model(torch.tensor([1.0]))`, 158-160, or any loss on z).  For dz[T,N,2] = dL/dz:
 *   grad_omega[N,Kb,2] = sum_t P[t]^T dz[t],  grad_a[N,2] = sum_t (1-t) dz[t],  grad_b[N,2] = sum_t t dz[t].
 * Fixed summation order, no atomics: repeated calls give the same bits.
 */
int vlg_spline_points_backward(int N, int T, int n_poly, const float* basis, const float* t,
                               const float* dz, float* grad_omega, float* grad_a, float* grad_b,
                               void* stream);

/* ---- spline fit to a poly-line ----------------------------------------------------------
 * omega[n] = argmin mean((lin + P_L omega - target_n)^2), the optimum that the reference's
 * LBFGS loop (src/init_splines_ensemble.py:175-192) iterates towards; end points are
 * target[0], target[L-1].  targets [N,Lmax,2] (row n uses the first lens[n] points),
 * lens int32 [N], omega out [N,Kb,2], ab out [N,2,2] (a then b).
 */
int vlg_fit_splines(int N, int Lmax, int n_poly, const float* targets, const int32_t* lens,
                    const float* basis, float* omega, float* ab, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VLG_H_ */
