"""Host-side mirror of the reference's interface for the geodesic hot path.

Same names and argument meaning as the reference where a counterpart exists:

  reference                                             here
  ---------------------------------------------------   -----------------------------------
  list(model.decoder)            (src/optimize.py:103)  DecoderEnsemble.from_state_dict(...)
  torch.stack([d(z).mean for d in decoders]) (50)       decoders(z), differentiable in z
  GeodesicSplineBatch(a,b,basis,omega,n_poly)   (13-35)  GeodesicSplineBatch (same signature)
  compute_energy_mc(model, decoders, t_vals, M) (38-75)  compute_energy_mc (same signature, +draws/seed)
  loss.sum().backward()                           (161)  autograd through compute_energy_mc and
                                                           GeodesicSplineBatch.forward (omega, a, b)
  optim.Adam([omega], lr) + the step loop     (153-162)  optimize_splines(model, decoders, t_vals, steps, ...)
  E over the draws of compute_energy_mc (M -> inf)       expected_curve_energy(decoders, model(t_vals)), differentiable
  compute_energy / compute_geodesic_lengths              compute_energy / compute_geodesic_lengths
     (src/single_decoder/optimize_energy_batched.py:42-57)
  construct_nullspace_basis      (optimize_energy.py:58)  construct_nullspace_basis
  build_entropy_weighted_graph's std field (init_splines_ensemble.py:47-54)  ensemble_std_norm

Everything heavy runs in the CUDA library through the ops in ``ops.py``; there is no CPU
fallback (CPU tensors raise).
"""
from __future__ import annotations

from typing import Optional, Sequence

import torch
from torch.autograd.function import once_differentiable

from . import _lib, ops

H = 128


class DecoderEnsemble:
    """K decoder MLPs 2 -> 128 -> 128 -> X repacked for the kernels (one device buffer).

    ``ens[:k]`` gives the first k decoders (``model.decoder[:k]``, src/eval.py:113); other
    slices are not supported, like in the reference's use."""

    def __init__(self, packed: torch.Tensor, K: int, X: int, k_active: Optional[int] = None):
        self.packed = packed
        self.K = K
        self.X = X
        self.k_active = K if k_active is None else k_active

    # ---- constructors -----------------------------------------------------------------
    @classmethod
    def from_arrays(cls, W1, b1, W2, b2, W3, b3, device) -> "DecoderEnsemble":
        dev = torch.device(device)
        if dev.type != "cuda":
            raise _lib.VlgError("DecoderEnsemble needs a CUDA device (vlg_b200 has no CPU path)")
        t = [torch.as_tensor(x, dtype=torch.float32).to(dev).contiguous() for x in (W1, b1, W2, b2, W3, b3)]
        K, Hd, X = t[0].shape[0], t[0].shape[1], t[4].shape[1]
        nbytes = ops.packed_decoders_bytes(K, Hd, X)
        packed = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        ops.pack_decoders(*t, packed)
        return cls(packed, K, X)

    @classmethod
    def from_state_dict(cls, state_dict, device, num_decoders: Optional[int] = None) -> "DecoderEnsemble":
        """EVAE checkpoint (experiment/model_seed*.pt): keys
        ``decoder.{i}.decoder_net.{0,2,4}.{weight,bias}`` (src/train.py:48-65,80-85)."""
        if num_decoders is None:
            ids = {int(k.split(".")[1]) for k in state_dict if k.startswith("decoder.") and k.split(".")[1].isdigit()}
            num_decoders = max(ids) + 1

        def grab(layer, what):
            return torch.stack([state_dict[f"decoder.{i}.decoder_net.{layer}.{what}"].float()
                                for i in range(num_decoders)])

        return cls.from_arrays(grab(0, "weight"), grab(0, "bias"), grab(2, "weight"), grab(2, "bias"),
                               grab(4, "weight"), grab(4, "bias"), device)

    @classmethod
    def from_state_dicts(cls, state_dicts, device, num_decoders: Optional[int] = None) -> "DecoderEnsemble":
        """Several EVAE checkpoints (e.g. the six seeds of the CoV study) packed back to back into ONE buffer:
        set s occupies decoders s * K .. s * K + K - 1; use with optimize_splines(decoder_base=..., k_active=...)."""
        parts = []
        for sd in state_dicts:
            if num_decoders is None:
                ids = {int(k.split(".")[1]) for k in sd if k.startswith("decoder.") and k.split(".")[1].isdigit()}
                num_decoders = max(ids) + 1
            parts.append([torch.stack([sd[f"decoder.{i}.decoder_net.{l}.{w}"].float() for i in range(num_decoders)])
                          for l, w in ((0, "weight"), (0, "bias"), (2, "weight"), (2, "bias"), (4, "weight"), (4, "bias"))])
        return cls.from_arrays(*[torch.cat([p[j] for p in parts]) for j in range(6)], device)

    @classmethod
    def from_single_vae_state_dict(cls, state_dict, device, out_dim: int = 50) -> "DecoderEnsemble":
        """Single VAE (src/artifacts/vae_best_seed*.pth): the decoder's last layer emits
        mean || log_std; ``.mean`` is rows 0:out_dim (src/single_decoder/vae.py:29-42)."""
        g = lambda l, w: state_dict[f"decoder.decoder_net.{l}.{w}"].float()
        return cls.from_arrays(g(0, "weight")[None], g(0, "bias")[None], g(2, "weight")[None], g(2, "bias")[None],
                               g(4, "weight")[None, :out_dim], g(4, "bias")[None, :out_dim], device)

    # ---- list-like view ---------------------------------------------------------------
    def __len__(self) -> int:
        return self.k_active

    def __getitem__(self, idx) -> "DecoderEnsemble":
        if isinstance(idx, slice) and idx.start in (None, 0) and idx.step in (None, 1):
            k = len(range(*idx.indices(self.k_active)))
            if k < 1:
                raise IndexError("empty decoder slice")
            return DecoderEnsemble(self.packed, self.K, self.X, k_active=k)
        raise IndexError("DecoderEnsemble supports only prefix slices ens[:k]")

    @property
    def device(self):
        return self.packed.device

    # ---- evaluation -------------------------------------------------------------------
    def __call__(self, z: torch.Tensor, precision: Optional[str] = None, check: bool = True) -> torch.Tensor:
        """Outputs of every active decoder at the latent points z [..., 2] (any float dtype): fp32 [K_active, ..., X],
        ``torch.stack([d(z).mean for d in decoders])`` of the reference (src/optimize.py:50,
        src/init_splines_ensemble.py:49).  E.g. ``decoders(model(t_vals))`` is its [K, T, N, X].

        Differentiable in z: with grad mode on and z.requires_grad, the backward runs vlg_decode_backward
        (dz = sum_k J_k(z)^T dx[k], no weight gradients, once differentiable).  precision=None is DEFAULT_PRECISION,
        with the fallbacks of the step kernels (more than 128 decoders, or one decoder in 'tf32' / 'f16': the fp32
        kernel).  check=True reads the status word back (one stream synchronisation) and raises VlgError on a
        non-finite output or gradient or a packed buffer that does not match its K / X."""
        if not isinstance(z, torch.Tensor) or not z.is_cuda:
            raise _lib.VlgError("DecoderEnsemble(z): z must be a CUDA tensor (vlg_b200 has no CPU path)")
        if z.dim() < 1 or z.shape[-1] != 2 or not z.is_floating_point():
            raise _lib.VlgError(f"DecoderEnsemble(z): z must be a float tensor [..., 2], got {z.dtype} {tuple(z.shape)}")
        prec = _resolve_precision(precision, self, 1)
        if torch.is_grad_enabled() and z.requires_grad:
            x = _Decode.apply(z, self, prec, check)
        else:
            x = _decode(self, z.detach().reshape(-1, 2).float().contiguous(), prec, check)
        return x.reshape(len(self), *z.shape[:-1], self.X)


def _refuse_untracked_grads(what: str, **tensors) -> None:
    """Gradients flow to omega, a and b only: refuse instead of leaving .grad of anything else at None."""
    if torch.is_grad_enabled():
        for name, x in tensors.items():
            if x.requires_grad:
                raise _lib.VlgError(f"{what}: no gradient with respect to {name} (only omega, a and b are differentiable)")


def _wants_grad(model) -> bool:
    return torch.is_grad_enabled() and (model.omega.requires_grad or model.a.requires_grad or model.b.requires_grad)


class _SplinePoints(torch.autograd.Function):
    """z = GeodesicSplineBatch.forward(t); backward by vlg_spline_points_backward (z is linear in omega, a, b)."""

    @staticmethod
    def forward(ctx, omega, a, b, basis, t, n_poly):
        z = torch.empty((t.shape[0], omega.shape[0], 2), dtype=torch.float32, device=omega.device)
        ops.spline_points(n_poly, a, b, omega, basis, t, z)
        ctx.save_for_backward(basis, t)
        ctx.n_poly, ctx.N, ctx.Kb = n_poly, omega.shape[0], omega.shape[1]
        return z

    @staticmethod
    @once_differentiable
    def backward(ctx, dz):
        basis, t = ctx.saved_tensors
        go = torch.empty((ctx.N, ctx.Kb, 2), dtype=torch.float32, device=dz.device)
        ga = torch.empty((ctx.N, 2), dtype=torch.float32, device=dz.device)
        gb = torch.empty_like(ga)
        ops.spline_points_backward(ctx.n_poly, basis, t, dz.contiguous().float(), go, ga, gb)
        return go, ga, gb, None, None, None


def _decode(decoders: DecoderEnsemble, z: torch.Tensor, prec: int, check: bool) -> torch.Tensor:
    """x [K_active, P, X] of the points z [P, 2] (fp32, contiguous)."""
    x = torch.empty((len(decoders), z.shape[0], decoders.X), dtype=torch.float32, device=z.device)
    if z.shape[0] == 0:
        return x
    ws = torch.empty(ops.DECODE_WORKSPACE_BYTES, dtype=torch.uint8, device=z.device)
    ops.decode(decoders.packed, decoders.K, decoders.X, len(decoders), z, x, prec, ws)
    if check:
        _raise_on_status(ws, "DecoderEnsemble")
    return x


def _decode_backward(decoders: DecoderEnsemble, z: torch.Tensor, dx: torch.Tensor, prec: int, check: bool) -> torch.Tensor:
    """dz [P, 2] = sum_k J_k(z)^T dx[k] for z [P, 2] and dx [K_active, P, X] (fp32, contiguous)."""
    dz = torch.empty((z.shape[0], 2), dtype=torch.float32, device=z.device)
    if z.shape[0] == 0:
        return dz
    ws = torch.empty(ops.DECODE_WORKSPACE_BYTES, dtype=torch.uint8, device=z.device)
    ops.decode_backward(decoders.packed, decoders.K, decoders.X, len(decoders), z, dx, dz, prec, ws)
    if check:
        _raise_on_status(ws, "DecoderEnsemble backward")
    return dz


class _Decode(torch.autograd.Function):
    """x = decoders(z); the backward recomputes the ReLU masks from z in vlg_decode_backward (no saved activations)."""

    @staticmethod
    def forward(ctx, z, decoders, prec, check):
        zf = z.detach().reshape(-1, 2).float().contiguous()
        ctx.save_for_backward(zf)
        ctx.decoders, ctx.prec, ctx.check, ctx.z_shape, ctx.z_dtype = decoders, prec, check, z.shape, z.dtype
        return _decode(decoders, zf, prec, check)

    @staticmethod
    def backward(ctx, dx):
        # once differentiable: the kernel forms dz only, so a graph of the backward (create_graph=True) cannot exist
        if torch.is_grad_enabled():
            raise _lib.VlgError("DecoderEnsemble: double backward is not supported (dz is once differentiable)")
        (zf,) = ctx.saved_tensors
        dz = _decode_backward(ctx.decoders, zf, dx.float().contiguous(), ctx.prec, ctx.check)
        return dz.reshape(ctx.z_shape).to(ctx.z_dtype), None, None, None


def _expected_energy(decoders: DecoderEnsemble, z: torch.Tensor, prec: int, check: bool, grad: bool):
    """(energy [N], dE/dz [T, N, 2] or None) of the curves z [T, N, 2] (fp32, contiguous)."""
    T, N = z.shape[0], z.shape[1]
    energy = torch.empty(N, dtype=torch.float32, device=z.device)
    dz = torch.empty_like(z) if grad else None
    if N == 0:
        return energy, dz
    ws = torch.empty(ops.expected_energy_workspace_bytes(N, T, decoders.X), dtype=torch.uint8, device=z.device)
    ops.expected_energy(decoders.packed, decoders.K, decoders.X, len(decoders), z, energy, dz, prec, ws)
    if check:
        _raise_on_status(ws, "expected_curve_energy")
    return energy, dz


class _ExpectedEnergy(torch.autograd.Function):
    """Expected energy [N] with the dE/dz one EnergyGrad launch formed next to it; the backward only scales dE/dz
    by the incoming dL/dE[n]."""

    @staticmethod
    def forward(ctx, z, decoders, prec, check):
        energy, dz = _expected_energy(decoders, z.detach().float().contiguous(), prec, check, grad=True)
        ctx.save_for_backward(dz)
        ctx.z_dtype = z.dtype
        return energy

    @staticmethod
    def backward(ctx, grad_e):
        # once differentiable: the kernel forms dE/dz only, so a graph of the backward (create_graph=True) cannot exist
        if torch.is_grad_enabled():
            raise _lib.VlgError("expected_curve_energy: double backward is not supported (dE/dz is once differentiable)")
        (dz,) = ctx.saved_tensors
        return (grad_e.to(torch.float32)[None, :, None] * dz).to(ctx.z_dtype), None, None, None


def expected_curve_energy(decoders: DecoderEnsemble, z: torch.Tensor, precision: Optional[str] = None,
                          check: bool = True) -> torch.Tensor:
    """Expected ensemble energy [N] of the curves z [T, N, 2] (any float dtype): the M -> infinity limit of
    compute_energy_mc (src/optimize.py:38-75), i.e. its expectation over independent uniform decoder pairs,
        E_n = sum_t ||mu_{t+1} - mu_t||^2 + sum_t c_t V_t,
    with mu_t / V_t the ensemble mean / variance of the decoder outputs at z_t and c_t the number of segments that
    touch point t.  Deterministic: ``torch.sqrt(expected_curve_energy(decoders, model(t_vals)))`` is the length the
    reference's MC value estimates.  z can be any point sequence (a spline's ``model(t_vals)``, a Dijkstra path).

    Differentiable in z: with grad mode on and z.requires_grad, ONE launch also forms dE/dz (once differentiable); a
    spline's omega, a and b get their gradients through model(t_vals).  precision=None is DEFAULT_PRECISION, with the
    fallbacks of DecoderEnsemble.__call__.  check=True reads the status word back (one stream synchronisation) and
    raises VlgError on a non-finite result or a packed buffer that does not match its K / X."""
    if not isinstance(z, torch.Tensor) or z.dim() != 3 or z.shape[-1] != 2 or not z.is_floating_point():
        raise _lib.VlgError(f"expected_curve_energy: z must be a float tensor [T, N, 2], got "
                            f"{getattr(z, 'dtype', type(z))} {tuple(getattr(z, 'shape', ()))}")
    if z.shape[0] < 2:
        raise _lib.VlgError(f"expected_curve_energy: a curve needs T >= 2 points, got T = {z.shape[0]}")
    if not z.is_cuda:
        raise _lib.VlgError("expected_curve_energy: z must be a CUDA tensor (vlg_b200 has no CPU path)")
    prec = _resolve_precision(precision, decoders, 1)
    if torch.is_grad_enabled() and z.requires_grad:
        return _ExpectedEnergy.apply(z, decoders, prec, check)
    return _expected_energy(decoders, z.detach().float().contiguous(), prec, check, grad=False)[0]


class _CurveEnergy(torch.autograd.Function):
    """Energy [N] with the gradients one vlg_curve_energy_grad launch formed next to it; the backward only
    scales them by the incoming dL/dE[n]."""

    @staticmethod
    def forward(ctx, omega, a, b, launch):
        energy, g_omega, g_a, g_b = launch()
        ctx.save_for_backward(g_omega, g_a, g_b)
        return energy

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_e):
        g_omega, g_a, g_b = ctx.saved_tensors
        ge = grad_e.to(torch.float32)
        need = ctx.needs_input_grad
        return (ge[:, None, None] * g_omega if need[0] else None, ge[:, None] * g_a if need[1] else None,
                ge[:, None] * g_b if need[2] else None, None)


class GeodesicSplineBatch:
    """Endpoint-constrained piecewise-cubic curves z_b(t) (src/optimize.py:13-35).
    Holds omega [N,Kb,2] (updated in place by optimize_splines) and the Adam state.

    omega, a and b are plain tensors; mark them ``requires_grad_()`` to differentiate forward(t) and
    compute_energy_mc with torch.autograd (the reference's nn.Parameter omega, src/optimize.py:20)."""

    def __init__(self, a, b, basis, omega, n_poly: int):
        self.a = a.contiguous().float()
        self.b = b.contiguous().float()
        self.basis = basis.contiguous().float()
        self.omega = omega.contiguous().float()
        self.n_poly = int(n_poly)
        self.adam_m = torch.zeros_like(self.omega)
        self.adam_v = torch.zeros_like(self.omega)
        self.step_count = 0

    def forward(self, t: torch.Tensor) -> torch.Tensor:
        t = t.contiguous().float()
        _refuse_untracked_grads("GeodesicSplineBatch.forward", basis=self.basis, t=t)
        if _wants_grad(self):
            return _SplinePoints.apply(self.omega, self.a, self.b, self.basis, t, self.n_poly)
        z = torch.empty((t.shape[0], self.omega.shape[0], 2), dtype=torch.float32, device=self.omega.device)
        ops.spline_points(self.n_poly, self.a, self.b, self.omega, self.basis, t, z)
        return z

    __call__ = forward


def _prep_draws(draws, N: int, steps: int, M: int, T: int, device, K_active: int) -> Optional[torch.Tensor]:
    """Reference layout [S,M,2,T-1,N] (any int dtype) -> kernel layout uint8 [N,S,M,2,T-1].
    Values must be decoder indices 0 <= d < K_active (torch.randint(0, K, ...), src/optimize.py:57-58)."""
    if draws is None:
        return None
    d = torch.as_tensor(draws)
    if d.dim() == 4:
        d = d[None]
    if tuple(d.shape) != (steps, M, 2, T - 1, N):
        raise _lib.VlgError(f"draws must have shape {(steps, M, 2, T - 1, N)}, got {tuple(d.shape)}")
    if d.is_floating_point() or d.dtype == torch.bool:
        raise _lib.VlgError(f"draws must be an integer tensor, got {d.dtype}")
    if d.numel():
        lo, hi = int(d.min()), int(d.max())
        if lo < 0 or hi >= K_active:
            raise _lib.VlgError(f"draws must lie in [0, {K_active}) for {K_active} active decoders, got [{lo}, {hi}]")
    return d.to(device=device, dtype=torch.uint8).permute(4, 0, 1, 2, 3).contiguous()


TC_MAX_M, TC_MAX_K = 2, 128   # tensor-core kernel (csrc/vlg_tc.cu): MC samples per block, decoder limit

# The ONE default arithmetic of the package, the drop-in CLIs (src/optimize.py, src/eval.py) and bench.py: the
# 3-term fp16 split in the forward GEMMs -- energies and lengths of a given curve are fp32-grade (1e-6) -- and
# single-term fp16 operands in the backward GEMMs (gradient to ~2.5e-4).  After 1000 free-running Adam steps on the
# benchmarked curves: median 1.0e-5, max 1.3e-4 against the reference's fp64 run where its own fp32 run has
# 8.3e-7 / 1.0e-4 (north-star bound 1e-3; tests/golden/config3_synth_1000.npz).  "f16x3" (all GEMMs 3-term) is the
# fp32-grade option, "f16" / "tf32" the 11-bit ones, "fp32" the CUDA-core kernel.
DEFAULT_PRECISION = "f16x3f"


def _resolve_precision(precision: Optional[str], decoders, M: int) -> int:
    """None -> DEFAULT_PRECISION.  Tensor-core precisions fall back to the fp32 CUDA-core kernel for shapes
    the tensor-core kernel is not built for (more than 128 decoders; any number of MC samples is fine: the kernel
    works through them in blocks of two); the single-term
    ones ('tf32', 'f16': 11-bit operands) also for a single active decoder, where they cannot resolve the tiny
    adjacent-point differences (SURVEY hard part 1; 'f16x3' can).  Still a GPU kernel -- there is no CPU
    path."""
    import warnings
    if precision is None:
        precision = DEFAULT_PRECISION
    if precision not in ops.PRECISIONS:
        raise _lib.VlgError(f"unknown precision {precision!r}; choose from {sorted(ops.PRECISIONS)}")
    if precision != "fp32" and len(decoders) > TC_MAX_K:
        warnings.warn(f"tensor-core kernel supports K <= {TC_MAX_K} decoders; using the fp32 kernel")
        precision = "fp32"
    if precision in ("tf32", "f16") and len(decoders) == 1:
        warnings.warn("single active decoder: 11-bit tensor-core operands cannot resolve adjacent-point "
                      "differences; using the fp32 kernel (f16x3 is the tensor-core option here)")
        precision = "fp32"
    return ops.PRECISIONS[precision]


def _workspace(model, decoders, T, M, precision):
    with torch.cuda.device(model.omega.device):   # grid sizing queries the SM count of the current device
        n = ops.workspace_bytes(model.omega.shape[0], T, model.n_poly, len(decoders), M, precision)
    return torch.empty(max(n, 256), dtype=torch.uint8, device=model.omega.device)


def _raise_on_status(ws: torch.Tensor, what: str) -> None:
    flags = ops.workspace_status(ws)
    if flags == 0:
        return
    why = []
    if flags & ops.STATUS_BAD_DRAW:
        why.append("an explicit draw was >= the number of active decoders")
    if flags & ops.STATUS_BAD_PACKED:
        why.append("the packed decoder buffer does not match its K / X")
    if flags & ops.STATUS_NONFINITE:
        why.append("non-finite energy or omega (with f16 / f16x3: a decoder activation or gradient beyond the "
                   "fp16 range 65504 -- use precision='tf32' or 'fp32')")
    raise _lib.VlgError(f"{what}: " + "; ".join(why))


def optimize_splines(model: GeodesicSplineBatch, decoders: DecoderEnsemble, t_vals: torch.Tensor, steps: int,
                     M: int = 2, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8,
                     penalty_weight: float = 1000.0, draws=None, seed: int = 0, curve_id0: int = 0,
                     precision: Optional[str] = None, return_trace: bool = False, check: bool = True,
                     stats: Optional[dict] = None, decoder_base=None, k_active: Optional[int] = None):
    """`steps` iterations of the loop at src/optimize.py:155-162 for every curve of `model`
    (fresh Adam state unless the model already stepped).  Returns the energy evaluated in the
    last step [N] (src/optimize.py:168) and, optionally, the per-step energies [steps,N].
    check=True reads the kernel's status word back after the launch (one stream synchronisation) and
    raises VlgError on a non-finite result (fp16 operand overflow) instead of returning garbage.
    stats: a dict that receives the launch's work counters ('items', 'rows'; tensor-core kernels).
    decoder_base / k_active: several weight sets in one launch -- curve n uses decoders
    decoder_base[n] .. decoder_base[n] + k_active - 1 of `decoders` (e.g. the ensembles of several training
    seeds packed with DecoderEnsemble.from_state_dicts; the CoV study of src/eval.py:90-128 in 10 launches)."""
    N = model.omega.shape[0]
    T = t_vals.shape[0]
    dev = model.omega.device
    if decoder_base is not None:
        if k_active is None:
            raise _lib.VlgError("decoder_base needs k_active (decoders per weight set)")
        decoder_base = torch.as_tensor(decoder_base)
        if tuple(decoder_base.shape) != (N,) or int(decoder_base.min()) < 0 or int(decoder_base.max()) + k_active > decoders.K:
            raise _lib.VlgError(f"decoder_base must be [N] with 0 <= base and base + {k_active} <= {decoders.K}")
        decoder_base = decoder_base.to(device=dev, dtype=torch.int32).contiguous()
        decoders = DecoderEnsemble(decoders.packed, decoders.K, decoders.X, k_active=k_active)
    prec = _resolve_precision(precision, decoders, M)
    energy = torch.empty(N, dtype=torch.float32, device=dev)
    trace = torch.empty((steps, N), dtype=torch.float32, device=dev) if return_trace else None
    if steps <= 0:
        raise _lib.VlgError("steps must be positive")
    ws = _workspace(model, decoders, T, M, prec)
    ops.optimize_steps(decoders.packed, decoders.K, decoders.X, len(decoders), model.n_poly, M, steps,
                       model.step_count, model.a, model.b,
                       model.omega, model.adam_m, model.adam_v, model.basis, t_vals.contiguous().float(),
                       _prep_draws(draws, N, steps, M, T, dev, len(decoders)), decoder_base, seed, curve_id0, lr, betas[0],
                       betas[1], eps, penalty_weight, energy, trace, prec, ws)
    model.step_count += steps
    if check:
        _raise_on_status(ws, "optimize_splines")
    if stats is not None:
        stats["items"], stats["rows"] = ops.workspace_counters(ws)
    return (energy, trace) if return_trace else energy


def compute_energy_mc(model: GeodesicSplineBatch, decoders: DecoderEnsemble, t_vals: torch.Tensor, M: int = 2,
                      draws=None, seed: int = 0, step: int = 0, curve_id0: int = 0, precision: str = "fp32",
                      return_length: bool = False, check: bool = True):
    """MC ensemble curve energy [N] (src/optimize.py:38-75).

    Differentiable in model.omega, model.a and model.b: when grad mode is on and any of them requires grad, ONE
    launch of the step kernel in gradient-output mode forms the energy and dE/d(omega), dE/da, dE/db (no penalty
    term), and the result carries a grad_fn whose backward only scales them (once differentiable).  Otherwise a
    forward-only launch.  The poly-line length (return_length) has no gradient."""
    N = model.omega.shape[0]
    T = t_vals.shape[0]
    prec = _resolve_precision(precision, decoders, M)
    dev = model.omega.device
    _refuse_untracked_grads("compute_energy_mc", basis=model.basis, t_vals=t_vals)
    grad = _wants_grad(model)
    if grad and return_length:
        raise _lib.VlgError("compute_energy_mc: return_length=True has no gradient; evaluate lengths under "
                            "torch.no_grad() (as src/single_decoder/optimize_energy_batched.py:42-49 does)")
    energy = torch.empty(N, dtype=torch.float32, device=dev)
    ws = _workspace(model, decoders, T, M, prec)
    args = (decoders.packed, decoders.K, decoders.X, len(decoders), model.n_poly, M, model.a.detach(),
            model.b.detach(), model.omega.detach(), model.basis, t_vals.contiguous().float(),
            _prep_draws(draws, N, 1, M, T, dev, len(decoders)), None, seed, curve_id0, step, energy)
    if grad:
        def launch():
            grads = (torch.empty_like(model.omega, dtype=torch.float32),
                     torch.empty((N, 2), dtype=torch.float32, device=dev),
                     torch.empty((N, 2), dtype=torch.float32, device=dev))
            ops.curve_energy_grad(*args, *grads, prec, ws)
            if check:
                _raise_on_status(ws, "compute_energy_mc")
            return (energy, *grads)

        return _CurveEnergy.apply(model.omega, model.a, model.b, launch)
    length = torch.empty(N, dtype=torch.float32, device=dev) if return_length else None
    ops.curve_energy(*args, length, prec, ws)
    if check:
        _raise_on_status(ws, "compute_energy_mc")
    return (energy, length) if return_length else energy


def compute_energy(spline: GeodesicSplineBatch, decoder: DecoderEnsemble, t_vals: torch.Tensor,
                   precision: str = "fp32") -> torch.Tensor:
    """Deterministic single-decoder energy (src/single_decoder/optimize_energy_batched.py:51-57)."""
    # one active decoder: every counter draw is 0, no draw tensor needed
    return compute_energy_mc(spline, decoder[:1], t_vals, M=1, precision=precision)


def compute_geodesic_lengths(spline: GeodesicSplineBatch, decoder: DecoderEnsemble, t_vals: torch.Tensor,
                             precision: str = "fp32") -> torch.Tensor:
    """Poly-line length in data space (src/single_decoder/optimize_energy_batched.py:42-49)."""
    return compute_energy_mc(spline, decoder[:1], t_vals, M=1, precision=precision, return_length=True)[1]


def optimize_single_decoder(model: GeodesicSplineBatch, decoder: DecoderEnsemble, t_vals: torch.Tensor,
                            steps: int = 500, lr: float = 1e-3, precision: Optional[str] = "f16x3"):
    """The loop of src/single_decoder/optimize_energy_batched.py:95-102 (deterministic energy).
    With a single active decoder every counter draw is 0, so no draw tensor is needed.  Default: f16x3 (all GEMMs
    3-term, fp32-grade on the tensor pipe; measured on the 64-curve x 500-step golden: median 1.9e-4,
    max 2.7e-3 against the reference's committed lengths, where its own CPU re-run has 1.3e-4 / 4.7e-3)."""
    return optimize_splines(model, decoder[:1], t_vals, steps, M=1, lr=lr, draws=None, precision=precision)


def ensemble_std_norm(decoders: DecoderEnsemble, grid: torch.Tensor) -> torch.Tensor:
    """|| std over decoders of f_k(grid) ||_2 (src/init_splines_ensemble.py:49-51)."""
    grid = grid.contiguous().float()
    out = torch.empty(grid.shape[0], dtype=torch.float32, device=grid.device)
    ops.ensemble_std_norm(decoders.packed, decoders.K, decoders.X, len(decoders), grid, out)
    return out


def fit_splines_to_paths(paths: Sequence[torch.Tensor], basis: torch.Tensor, n_poly: int, device):
    """Least-squares spline fit to poly-lines (src/init_splines_ensemble.py:172-193), batched.
    Returns (a [N,2], b [N,2], omega [N,Kb,2])."""
    N = len(paths)
    Lmax = max(int(p.shape[0]) for p in paths)
    tg = torch.zeros((N, Lmax, 2), dtype=torch.float32)
    lens = torch.zeros(N, dtype=torch.int32)
    for i, p in enumerate(paths):
        tg[i, : p.shape[0]] = torch.as_tensor(p, dtype=torch.float32)
        lens[i] = p.shape[0]
    tg, lens = tg.to(device), lens.to(device)
    basis = basis.to(device).contiguous().float()
    omega = torch.empty((N, n_poly + 1, 2), dtype=torch.float32, device=device)
    ab = torch.empty((N, 2, 2), dtype=torch.float32, device=device)
    ops.fit_splines(n_poly, tg, lens, basis, omega, ab)
    return ab[:, 0].contiguous(), ab[:, 1].contiguous(), omega


def construct_nullspace_basis(n_poly: int, device="cpu"):
    """Orthonormal basis of the spline coefficients that keep offset(0)=offset(1)=0 and C0/C1/C2
    continuity at the inner knots (src/single_decoder/optimize_energy.py:58-102).  fp64 SVD + QR on
    the host, returned as fp32.  NOTE the basis is not unique across LAPACK builds (SURVEY hard
    part 7): when consuming existing omegas always take the basis stored in the spline file."""
    n = int(n_poly)
    rows = []
    first = torch.zeros(4 * n, dtype=torch.float64)
    first[0] = 1.0
    last = torch.zeros(4 * n, dtype=torch.float64)
    last[4 * n - 4:] = 1.0
    rows += [first, last]
    # value / first / second derivative of (1, u, u^2, u^3) at u=1 (left piece) and u=0 (right piece)
    left = torch.tensor([[1, 1, 1, 1], [0, 1, 2, 3], [0, 0, 2, 6]], dtype=torch.float64)
    right = torch.tensor([[1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 2, 0]], dtype=torch.float64)
    for knot in range(n - 1):
        for order in range(3):
            r = torch.zeros(4 * n, dtype=torch.float64)
            r[4 * knot: 4 * knot + 4] = left[order]
            r[4 * knot + 4: 4 * knot + 8] = -right[order]
            rows.append(r)
    C = torch.stack(rows)
    _, S, Vh = torch.linalg.svd(C, full_matrices=True)
    rank = int((S > 1e-10 * S[0]).sum())
    null = Vh.T[:, rank:].contiguous()
    basis = torch.linalg.qr(null)[0]
    return basis.to(torch.float32).to(device), C.to(torch.float32).to(device)
