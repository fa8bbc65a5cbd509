"""torch custom ops: thin shims from tensors to the C ABI (include/vlg.h).

Each op checks dtype / contiguity / device, passes ``data_ptr()`` and the current CUDA
stream, and raises on a non-zero return code.  No CPU implementation is registered: calling
these with CPU tensors is an error, by design.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib

PRECISIONS = {"fp32": 0, "tf32": 1, "f16x3": 2, "tf32x3": 2, "f16": 3, "f16x3f": 4}


def _chk(x: Optional[torch.Tensor], name: str, dtype=torch.float32, shape=None):
    if x is None:
        return 0
    if not x.is_cuda:
        raise _lib.VlgError(f"{name} must be a CUDA tensor (vlg_b200 has no CPU path)")
    if x.dtype != dtype:
        raise _lib.VlgError(f"{name} must be {dtype}, got {x.dtype}")
    if not x.is_contiguous():
        raise _lib.VlgError(f"{name} must be contiguous")
    if shape is not None and tuple(x.shape) != tuple(shape):
        raise _lib.VlgError(f"{name} must have shape {tuple(shape)}, got {tuple(x.shape)}")
    return x.data_ptr()


def _stream(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def packed_decoders_bytes(K: int, H: int, X: int) -> int:
    n = _lib.load().vlg_packed_decoders_bytes(K, H, X)
    if n == 0:
        raise _lib.VlgError(f"unsupported decoder shape K={K} H={H} X={X} (need H=128, X<=52, K<=254)")
    return n


@torch.library.custom_op("vlg::pack_decoders", mutates_args=("packed",))
def pack_decoders(W1: torch.Tensor, b1: torch.Tensor, W2: torch.Tensor, b2: torch.Tensor,
                  W3: torch.Tensor, b3: torch.Tensor, packed: torch.Tensor) -> None:
    K, H = W1.shape[0], W1.shape[1]
    X = W3.shape[1]
    ptrs = [_chk(W1, "W1", shape=(K, H, 2)), _chk(b1, "b1", shape=(K, H)),
            _chk(W2, "W2", shape=(K, H, H)), _chk(b2, "b2", shape=(K, H)),
            _chk(W3, "W3", shape=(K, X, H)), _chk(b3, "b3", shape=(K, X))]
    if packed.numel() * packed.element_size() < packed_decoders_bytes(K, H, X):
        raise _lib.VlgError("packed buffer too small")
    pp = _chk(packed, "packed", dtype=packed.dtype)
    with torch.cuda.device(W1.device):
        _lib.check(_lib.load().vlg_pack_decoders(*ptrs, K, H, X, pp, _stream(W1)), "vlg_pack_decoders")


def workspace_bytes(N: int, T: int, n_poly: int, K_active: int, M: int, precision: int) -> int:
    return _lib.load().vlg_workspace_bytes(N, T, n_poly, K_active, M, precision)


STATUS_BAD_DRAW, STATUS_NONFINITE, STATUS_BAD_PACKED = 1, 2, 4


def workspace_counters(workspace: torch.Tensor):
    """(items, rows) executed by the last tensor-core launch that used `workspace` (synchronises)."""
    import ctypes
    out = (ctypes.c_ulonglong * 2)()
    with torch.cuda.device(workspace.device):
        _lib.check(_lib.load().vlg_workspace_counters(_chk(workspace, "workspace", dtype=torch.uint8), out,
                                                      _stream(workspace)), "vlg_workspace_counters")
    return int(out[0]), int(out[1])


def workspace_status(workspace: torch.Tensor) -> int:
    """VLG_STATUS_* flags of the last step-kernel or decode launch that used `workspace` (synchronises the stream)."""
    import ctypes
    flags = ctypes.c_int(0)
    with torch.cuda.device(workspace.device):
        rc = _lib.load().vlg_workspace_status(_chk(workspace, "workspace", dtype=torch.uint8), ctypes.byref(flags),
                                              _stream(workspace))
    if rc not in (0, -6):
        _lib.check(rc, "vlg_workspace_status")
    return flags.value


def _step_args(packed, k_total, x_dim, k_active, n_poly, M, steps, a, b, omega, basis, t, draws, decoder_base, seed,
               curve_id0, workspace):
    """Checks the tensors the three step ops share.  Returns their C-ABI arguments in the runs the entry points
    take them: (packed .. M), (a, b, omega), (basis .. curve_id0) and (workspace, its bytes, stream)."""
    N, Kb = omega.shape[0], omega.shape[1]
    T = t.shape[0]
    if Kb != n_poly + 1:
        raise _lib.VlgError(f"omega has Kb={Kb}, expected n_poly+1={n_poly + 1}")
    head = [_chk(packed, "packed", dtype=packed.dtype), k_total, x_dim, k_active, N, T, n_poly, M]
    curve = [_chk(a, "a", shape=(N, 2)), _chk(b, "b", shape=(N, 2)), _chk(omega, "omega", shape=(N, Kb, 2))]
    tail = [_chk(basis, "basis", shape=(4 * n_poly, Kb)), _chk(t, "t", shape=(T,)),
            _chk(draws, "draws", dtype=torch.uint8, shape=(N, steps, M, 2, T - 1)),
            _chk(decoder_base, "decoder_base", dtype=torch.int32, shape=(N,)), seed & 0xFFFFFFFFFFFFFFFF, curve_id0]
    ws = [_chk(workspace, "workspace", dtype=torch.uint8), workspace.numel() if workspace is not None else 0,
          _stream(omega)]
    return head, curve, tail, ws


@torch.library.custom_op("vlg::optimize_steps",
                         mutates_args=("omega", "adam_m", "adam_v", "energy_last", "energy_trace", "workspace"))
def optimize_steps(packed: torch.Tensor, k_total: int, x_dim: int, k_active: int, n_poly: int, M: int, steps: int, step0: int,
                   a: torch.Tensor, b: torch.Tensor, omega: torch.Tensor, adam_m: torch.Tensor,
                   adam_v: torch.Tensor, basis: torch.Tensor, t: torch.Tensor,
                   draws: Optional[torch.Tensor], decoder_base: Optional[torch.Tensor], seed: int, curve_id0: int,
                   lr: float, beta1: float,
                   beta2: float, eps: float, penalty_w: float, energy_last: torch.Tensor,
                   energy_trace: Optional[torch.Tensor], precision: int,
                   workspace: Optional[torch.Tensor]) -> None:
    head, curve, tail, ws = _step_args(packed, k_total, x_dim, k_active, n_poly, M, steps, a, b, omega, basis, t, draws,
                                       decoder_base, seed, curve_id0, workspace)
    N = omega.shape[0]
    args = [*head, steps, step0, *curve, _chk(adam_m, "adam_m", shape=omega.shape),
            _chk(adam_v, "adam_v", shape=omega.shape), *tail, lr, beta1, beta2, eps, penalty_w,
            _chk(energy_last, "energy_last", shape=(N,)), _chk(energy_trace, "energy_trace", shape=(steps, N)),
            precision, *ws]
    with torch.cuda.device(omega.device):
        _lib.check(_lib.load().vlg_optimize_steps(*args), "vlg_optimize_steps")


@torch.library.custom_op("vlg::curve_energy", mutates_args=("energy", "length", "workspace"))
def curve_energy(packed: torch.Tensor, k_total: int, x_dim: int, k_active: int, n_poly: int, M: int, a: torch.Tensor,
                 b: torch.Tensor, omega: torch.Tensor, basis: torch.Tensor, t: torch.Tensor,
                 draws: Optional[torch.Tensor], decoder_base: Optional[torch.Tensor], seed: int, curve_id0: int, step: int,
                 energy: torch.Tensor, length: Optional[torch.Tensor], precision: int,
                 workspace: Optional[torch.Tensor]) -> None:
    head, curve, tail, ws = _step_args(packed, k_total, x_dim, k_active, n_poly, M, 1, a, b, omega, basis, t, draws,
                                       decoder_base, seed, curve_id0, workspace)
    N = omega.shape[0]
    args = [*head, *curve, *tail, step, _chk(energy, "energy", shape=(N,)), _chk(length, "length", shape=(N,)),
            precision, *ws]
    with torch.cuda.device(omega.device):
        _lib.check(_lib.load().vlg_curve_energy(*args), "vlg_curve_energy")


@torch.library.custom_op("vlg::curve_energy_grad",
                         mutates_args=("energy", "grad_omega", "grad_a", "grad_b", "workspace"))
def curve_energy_grad(packed: torch.Tensor, k_total: int, x_dim: int, k_active: int, n_poly: int, M: int,
                      a: torch.Tensor, b: torch.Tensor, omega: torch.Tensor, basis: torch.Tensor, t: torch.Tensor,
                      draws: Optional[torch.Tensor], decoder_base: Optional[torch.Tensor], seed: int, curve_id0: int,
                      step: int, energy: torch.Tensor, grad_omega: torch.Tensor, grad_a: torch.Tensor,
                      grad_b: torch.Tensor, precision: int, workspace: Optional[torch.Tensor]) -> None:
    head, curve, tail, ws = _step_args(packed, k_total, x_dim, k_active, n_poly, M, 1, a, b, omega, basis, t, draws,
                                       decoder_base, seed, curve_id0, workspace)
    N = omega.shape[0]
    args = [*head, *curve, *tail, step, _chk(energy, "energy", shape=(N,)),
            _chk(grad_omega, "grad_omega", shape=omega.shape), _chk(grad_a, "grad_a", shape=(N, 2)),
            _chk(grad_b, "grad_b", shape=(N, 2)), precision, *ws]
    with torch.cuda.device(omega.device):
        _lib.check(_lib.load().vlg_curve_energy_grad(*args), "vlg_curve_energy_grad")


@torch.library.custom_op("vlg::ensemble_std_norm", mutates_args=("out",))
def ensemble_std_norm(packed: torch.Tensor, k_total: int, x_dim: int, k_active: int, grid: torch.Tensor,
                      out: torch.Tensor) -> None:
    G = grid.shape[0]
    with torch.cuda.device(grid.device):
        _lib.check(_lib.load().vlg_ensemble_std_norm(_chk(packed, "packed", dtype=packed.dtype), k_total, x_dim,
                                                     k_active, G,
                                                     _chk(grid, "grid", shape=(G, 2)),
                                                     _chk(out, "out", shape=(G,)), _stream(grid)),
                   "vlg_ensemble_std_norm")


DECODE_WORKSPACE_BYTES = 256   # VLG_DECODE_WORKSPACE_BYTES


@torch.library.custom_op("vlg::decode", mutates_args=("x", "workspace"))
def decode(packed: torch.Tensor, k_total: int, x_dim: int, k_active: int, z: torch.Tensor, x: torch.Tensor,
           precision: int, workspace: torch.Tensor) -> None:
    P = z.shape[0]
    with torch.cuda.device(z.device):
        _lib.check(_lib.load().vlg_decode(_chk(packed, "packed", dtype=packed.dtype), k_total, x_dim, k_active, P,
                                          _chk(z, "z", shape=(P, 2)), _chk(x, "x", shape=(k_active, P, x_dim)),
                                          precision, _chk(workspace, "workspace", dtype=torch.uint8), workspace.numel(),
                                          _stream(z)), "vlg_decode")


@torch.library.custom_op("vlg::decode_backward", mutates_args=("dz", "workspace"))
def decode_backward(packed: torch.Tensor, k_total: int, x_dim: int, k_active: int, z: torch.Tensor, dx: torch.Tensor,
                    dz: torch.Tensor, precision: int, workspace: torch.Tensor) -> None:
    P = z.shape[0]
    with torch.cuda.device(z.device):
        _lib.check(_lib.load().vlg_decode_backward(_chk(packed, "packed", dtype=packed.dtype), k_total, x_dim,
                                                   k_active, P, _chk(z, "z", shape=(P, 2)),
                                                   _chk(dx, "dx", shape=(k_active, P, x_dim)),
                                                   _chk(dz, "dz", shape=(P, 2)), precision,
                                                   _chk(workspace, "workspace", dtype=torch.uint8), workspace.numel(),
                                                   _stream(z)), "vlg_decode_backward")


def expected_energy_workspace_bytes(N: int, T: int, X: int) -> int:
    n = _lib.load().vlg_expected_energy_workspace_bytes(N, T, X)
    if n == 0:
        raise _lib.VlgError(f"unsupported expected-energy shape N={N} T={T} X={X} (need N >= 1, T >= 2, T*N < 2^31, X <= 52)")
    return n


@torch.library.custom_op("vlg::expected_energy", mutates_args=("energy", "grad_z", "workspace"))
def expected_energy(packed: torch.Tensor, k_total: int, x_dim: int, k_active: int, z: torch.Tensor,
                    energy: torch.Tensor, grad_z: Optional[torch.Tensor], precision: int,
                    workspace: torch.Tensor) -> None:
    T, N = z.shape[0], z.shape[1]
    with torch.cuda.device(z.device):
        _lib.check(_lib.load().vlg_expected_energy(_chk(packed, "packed", dtype=packed.dtype), k_total, x_dim, k_active,
                                                   N, T, _chk(z, "z", shape=(T, N, 2)),
                                                   _chk(energy, "energy", shape=(N,)),
                                                   _chk(grad_z, "grad_z", shape=(T, N, 2)), precision,
                                                   _chk(workspace, "workspace", dtype=torch.uint8), workspace.numel(),
                                                   _stream(z)), "vlg_expected_energy")


@torch.library.custom_op("vlg::spline_points", mutates_args=("z",))
def spline_points(n_poly: int, a: torch.Tensor, b: torch.Tensor, omega: torch.Tensor, basis: torch.Tensor,
                  t: torch.Tensor, z: torch.Tensor) -> None:
    N, Kb = omega.shape[0], omega.shape[1]
    T = t.shape[0]
    with torch.cuda.device(omega.device):
        _lib.check(_lib.load().vlg_spline_points(N, T, n_poly, _chk(a, "a", shape=(N, 2)),
                                                 _chk(b, "b", shape=(N, 2)),
                                                 _chk(omega, "omega", shape=(N, Kb, 2)),
                                                 _chk(basis, "basis", shape=(4 * n_poly, Kb)),
                                                 _chk(t, "t", shape=(T,)), _chk(z, "z", shape=(T, N, 2)),
                                                 _stream(omega)), "vlg_spline_points")


@torch.library.custom_op("vlg::spline_points_backward", mutates_args=("grad_omega", "grad_a", "grad_b"))
def spline_points_backward(n_poly: int, basis: torch.Tensor, t: torch.Tensor, dz: torch.Tensor,
                           grad_omega: torch.Tensor, grad_a: torch.Tensor, grad_b: torch.Tensor) -> None:
    N, Kb = grad_omega.shape[0], grad_omega.shape[1]
    T = t.shape[0]
    with torch.cuda.device(dz.device):
        _lib.check(_lib.load().vlg_spline_points_backward(N, T, n_poly,
                                                          _chk(basis, "basis", shape=(4 * n_poly, Kb)),
                                                          _chk(t, "t", shape=(T,)), _chk(dz, "dz", shape=(T, N, 2)),
                                                          _chk(grad_omega, "grad_omega", shape=(N, Kb, 2)),
                                                          _chk(grad_a, "grad_a", shape=(N, 2)),
                                                          _chk(grad_b, "grad_b", shape=(N, 2)), _stream(dz)),
                   "vlg_spline_points_backward")


@torch.library.custom_op("vlg::fit_splines", mutates_args=("omega", "ab"))
def fit_splines(n_poly: int, targets: torch.Tensor, lens: torch.Tensor, basis: torch.Tensor,
                omega: torch.Tensor, ab: torch.Tensor) -> None:
    N, Lmax = targets.shape[0], targets.shape[1]
    Kb = n_poly + 1
    with torch.cuda.device(targets.device):
        _lib.check(_lib.load().vlg_fit_splines(N, Lmax, n_poly, _chk(targets, "targets", shape=(N, Lmax, 2)),
                                               _chk(lens, "lens", dtype=torch.int32, shape=(N,)),
                                               _chk(basis, "basis", shape=(4 * n_poly, Kb)),
                                               _chk(omega, "omega", shape=(N, Kb, 2)),
                                               _chk(ab, "ab", shape=(N, 2, 2)), _stream(targets)),
                   "vlg_fit_splines")
