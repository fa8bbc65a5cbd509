"""Differentiable curve energy: vlg_curve_energy_grad (energy and dE/d(omega), dE/da, dE/db from one step-kernel
launch), vlg_spline_points_backward, and autograd through compute_energy_mc / GeodesicSplineBatch.forward.

The CPU tests check the C ABI without a device; the GPU tests compare against the fp64 oracle and fp64
torch.autograd through oracle.torch_port on recorded draws."""
import ctypes
import functools

import numpy as np
import pytest
import torch

from oracle import geodesic_oracle as O
from tests import helpers as Hh

MC_CASES = ["ens_seed12_euclid", "ens_seed12_entropy", "ens_seed12_cov_k3", "synth_np8_T256", "synth_np4_T130"]
PRECISIONS = ["fp32", "f16x3", "f16x3f", "f16", "tf32"]
# relative error bound of the gradient per arithmetic (fp32: the bar of the optimiser's first-Adam-moment test).
# The 11-bit modes (f16, tf32) reach 1.5e-2 on dE/domega and 4.9e-2 on dE/da of ens_seed12_entropy, whose gradient is
# a small difference of large per-point terms; the optimiser's own step gradient has the same bits (see
# test_same_numbers_as_the_optimiser_step).
GRAD_TOL = {"fp32": 2e-5, "f16x3": 2e-4, "f16x3f": 5e-3, "f16": 6e-2, "tf32": 6e-2}


# ------------------------------------------------------------------ CPU ------------------------------------------

def test_header_declares_and_library_exports_the_gradient_entries(built_lib):
    from tests.test_cabi import declared_functions
    names = declared_functions()
    lib = ctypes.CDLL(str(built_lib))
    for name in ("vlg_curve_energy_grad", "vlg_spline_points_backward"):
        assert name in names
        assert hasattr(lib, name)


def test_gradient_entries_reject_bad_arguments_before_any_device_call(built_lib):
    from vlg_b200 import _lib
    lib = _lib.load()
    p = ctypes.c_void_p(16)   # never dereferenced: validation fails first
    # vlg_curve_energy_grad: a null input or a null output
    args = [p, 10, 50, 10, 4, 2000, 4, 2, p, p, p, p, p, None, None, 0, 0, 0, p, p, p, p, 0, p, 1 << 20, None]
    for i in (8, 9, 10, 11, 12, 18, 19, 20, 21):
        bad = list(args)
        bad[i] = None
        assert lib.vlg_curve_energy_grad(*bad) == -1, i
    bad = list(args)
    bad[17] = -1                                                  # step < 0
    assert lib.vlg_curve_energy_grad(*bad) == -1
    # vlg_spline_points_backward: null pointers, non-positive sizes
    ok = [3, 10, 4, p, p, p, p, p, p, None]
    for i in range(3, 9):
        bad = list(ok)
        bad[i] = None
        assert lib.vlg_spline_points_backward(*bad) == -1, i
    for i in range(3):
        bad = list(ok)
        bad[i] = 0
        assert lib.vlg_spline_points_backward(*bad) == -1, i


# ------------------------------------------------------------------ GPU ------------------------------------------

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def vlg(built_lib):
    import vlg_b200
    assert torch.cuda.is_available(), "GPU tests need a B200"
    return vlg_b200


def make_model(vlg, g, dev="cuda"):
    return vlg.GeodesicSplineBatch(torch.tensor(g["a"], device=dev), torch.tensor(g["b"], device=dev),
                                   torch.tensor(g["basis"], device=dev), torch.tensor(g["omega_init"], device=dev),
                                   int(g["n_poly"]))


def make_decoders(vlg, g, K, dev="cuda"):
    arrs = Hh.decoder_arrays(g)
    return vlg.DecoderEnsemble.from_arrays(*[arrs[k] for k in Hh.DEC_KEYS], dev)[:K]


def energy_grad(vlg, model, dec, t, M, prec, draws=None, seed=0, curve_id0=0, step=0, decoder_base=None,
                outs=None):
    """One vlg_curve_energy_grad launch through the op -> (energy, dE/domega, dE/da, dE/db, status flags)."""
    from vlg_b200 import api, ops
    N = model.omega.shape[0]
    T = t.shape[0]
    code = ops.PRECISIONS[prec]
    if outs is None:
        outs = (torch.empty(N, device="cuda"), torch.empty_like(model.omega), torch.empty(N, 2, device="cuda"),
                torch.empty(N, 2, device="cuda"))
    ws = api._workspace(model, dec, T, M, code)
    d = api._prep_draws(draws, N, 1, M, T, "cuda", len(dec)) if draws is not None and draws.dtype != torch.uint8 \
        else draws
    ops.curve_energy_grad(dec.packed, dec.K, dec.X, len(dec), model.n_poly, M, model.a, model.b, model.omega,
                          model.basis, t, d, decoder_base, seed, curve_id0, step, *outs, code, ws)
    return (*outs, ops.workspace_status(ws))


@functools.lru_cache(maxsize=None)
def fp64_reference(tag):
    """dE/domega from the hand-derived fp64 oracle (no penalty), and dE/domega, da, db from fp64 torch.autograd
    through oracle.torch_port, on the golden's step-0 draws."""
    from oracle import torch_port as TP
    g = Hh.load(tag)
    K, T = int(g["K"]), int(g["T"])
    n_poly = int(g["n_poly"])
    d0 = Hh.regen_draws(g)[0]                       # [M,2,T-1,N]
    a, b, om, basis = (g[k].astype(np.float64) for k in ("a", "b", "omega_init", "basis"))
    t = Hh.tgrid(T).astype(np.float64)            # the fp32 grid the kernels see
    decs = Hh.decoder_list(Hh.decoder_arrays(g), K, np.float64)
    E, grad, end_err = O.energy_mc_grad(a, b, om, basis, t, n_poly, decs, d0, penalty_w=0.0)
    # cross-check: the golden's loss gradient minus its penalty term (synth_np8_T256's golden energy and gradient sit
    # 4e-8 / 3e-8 from the oracle on the stored arrays; the others agree to 1e-15)
    P1 = O.design_matrix(basis, t[-1:], n_poly)[0]
    assert Hh.relerr(grad + 2000.0 * end_err[:, None, :] * P1[None, :, None], g["grad0_f64"]) < 1e-7

    ta = torch.tensor(a, requires_grad=True)
    tb = torch.tensor(b, requires_grad=True)
    sb = TP.SplineBatch(ta, tb, torch.tensor(basis), torch.tensor(om), n_poly)
    nets = [TP.make_decoder(w).double() for w in decs]
    e = TP.energy_mc(sb, nets, torch.tensor(t), d0.shape[0], torch.as_tensor(d0))
    e.sum().backward()
    return dict(E=E, grad=grad, ga=ta.grad.numpy(), gb=tb.grad.numpy(), gom_torch=sb.omega.grad.numpy())


def _case(vlg, tag, prec):
    g = Hh.load(tag)
    K, T, M = int(g["K"]), int(g["T"]), int(g["M"])
    model = make_model(vlg, g)
    dec = make_decoders(vlg, g, K)
    t = torch.linspace(0, 1, T, device="cuda")
    draws = torch.as_tensor(Hh.regen_draws(g)[:1])
    return g, model, dec, t, M, draws


@gpu
@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("tag", MC_CASES)
def test_gradient_matches_fp64_oracle(vlg, tag, prec):
    g, model, dec, t, M, draws = _case(vlg, tag, prec)
    ref = fp64_reference(tag)
    E, gom, _, _, flags = energy_grad(vlg, model, dec, t, M, prec, draws)
    assert flags == 0
    err = Hh.relerr(gom.cpu().numpy(), ref["grad"])
    print(f"{tag} {prec}: dE/domega relerr {err:.2e}, energy relerr {Hh.relerr(E.cpu().numpy(), ref['E']):.2e}")
    assert err < GRAD_TOL[prec]
    assert Hh.relerr(ref["gom_torch"], ref["grad"]) < 1e-10     # the two fp64 references agree


@gpu
@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("tag", MC_CASES)
def test_endpoint_gradients_match_fp64_autograd(vlg, tag, prec):
    g, model, dec, t, M, draws = _case(vlg, tag, prec)
    ref = fp64_reference(tag)
    _, _, ga, gb, flags = energy_grad(vlg, model, dec, t, M, prec, draws)
    assert flags == 0
    ea, eb = Hh.relerr(ga.cpu().numpy(), ref["ga"]), Hh.relerr(gb.cpu().numpy(), ref["gb"])
    print(f"{tag} {prec}: dE/da relerr {ea:.2e}, dE/db relerr {eb:.2e}")
    assert ea < GRAD_TOL[prec] and eb < GRAD_TOL[prec]


@gpu
@pytest.mark.parametrize("prec", PRECISIONS)
def test_same_numbers_as_the_optimiser_step(vlg, prec):
    """Energy bit-identical to optimize_splines' trace[0]; dE/domega = adam_m / (1 - beta1) minus the penalty."""
    g, model, dec, t, M, draws = _case(vlg, "ens_seed12_euclid", prec)
    E, gom, _, _, _ = energy_grad(vlg, model, dec, t, M, prec, draws)
    opt_model = make_model(vlg, g)
    _, trace = vlg.optimize_splines(opt_model, dec, t, 1, M=M, draws=draws.numpy(), precision=prec, return_trace=True)
    assert torch.equal(E, trace[0])
    n_poly = int(g["n_poly"])
    err = (model(t[-1:])[0] - model.b).double().cpu().numpy()
    P1 = O.design_matrix(g["basis"].astype(np.float64), Hh.tgrid(int(g["T"])).astype(np.float64)[-1:], n_poly)[0]
    pen = 2000.0 * err[:, None, :] * P1[None, :, None]
    g_opt = opt_model.adam_m.double().cpu().numpy() / (1 - 0.9) - pen
    assert Hh.relerr(gom.cpu().numpy(), g_opt) < 1e-6
    if prec in ("fp32", "f16x3", "f16x3f"):
        E_fwd = vlg.compute_energy_mc(model, dec, t, M=M, draws=draws.numpy(), precision=prec)
        assert Hh.relerr(E.cpu().numpy(), E_fwd.cpu().numpy()) < 1e-6


@gpu
def test_reference_loop_runs_unchanged(vlg):
    """src/optimize.py:155-162 verbatim on vlg_b200: torch.optim.Adam, the energy plus the end-point penalty
    through model(t), loss.sum().backward(), step()."""
    g = Hh.load("ens_seed12_euclid")
    K, T, M, S = int(g["K"]), int(g["T"]), int(g["M"]), int(g["steps"])
    draws = Hh.regen_draws(g)[:S]
    dec = make_decoders(vlg, g, K)
    t = torch.linspace(0, 1, T, device="cuda")

    def run(model, precision, each_step=None):
        model.omega.requires_grad_(True)
        optimizer = torch.optim.Adam([model.omega], lr=1e-3)
        energies = []
        for s in range(S):
            optimizer.zero_grad()
            energy = vlg.compute_energy_mc(model, dec, t, M, draws=draws[s], precision=precision)
            z_end = model(t[-1:])
            loss = energy + 1000 * ((z_end - model.b) ** 2).sum(-1)
            loss.sum().backward()
            optimizer.step()
            energies.append(energy.detach().cpu().numpy())
            if each_step:
                each_step(s, model.omega.detach())
        return np.stack(energies)

    model = make_model(vlg, g)
    energies = run(model, "fp32")
    rel = np.abs(energies / g["energy_f64"] - 1).max()
    print(f"reference loop fp32: energy rel err {rel:.2e}")
    assert rel < 5e-6
    assert np.abs(model.omega.detach().cpu().numpy() - g["omega_f64"]).max() < 5e-6

    # the same loop in the default precision against the fused optimiser, step by step
    fused = make_model(vlg, g)
    gaps = []

    def compare(s, omega):
        vlg.optimize_splines(fused, dec, t, 1, M=M, draws=draws[s:s + 1])
        gaps.append(float((omega - fused.omega).abs().max()))

    run(make_model(vlg, g), None, compare)
    print(f"reference loop default precision vs optimize_splines: max |d omega| per step {gaps}")
    assert max(gaps) < 1e-6


@gpu
def test_single_decoder_loop_with_compute_energy(vlg):
    """The single-decoder loop (src/single_decoder/optimize_energy_batched.py:95-102) written with torch.optim and
    compute_energy, with the end-point penalty optimize_single_decoder applies, against optimize_single_decoder."""
    g = Hh.load("single_seed123")
    dec = make_decoders(vlg, g, 1)
    t = torch.linspace(0, 1, 2000, device="cuda")
    S = 3
    spline = make_model(vlg, g)
    spline.omega.requires_grad_(True)
    optimizer = torch.optim.Adam([spline.omega], lr=1e-3)
    for _ in range(S):
        optimizer.zero_grad()
        energy = vlg.compute_energy(spline, dec, t, precision="fp32")
        z_end = spline(t[-1:])
        loss = energy + 1000 * ((z_end - spline.b) ** 2).sum(-1)
        loss.sum().backward()
        optimizer.step()
    fused = make_model(vlg, g)
    vlg.optimize_single_decoder(fused, dec, t, steps=S, precision="fp32")
    gap = float((spline.omega.detach() - fused.omega).abs().max())
    print(f"single-decoder loop vs optimize_single_decoder: max |d omega| {gap:.2e}")
    assert gap < 1e-6


def _random_case(N, K, n_poly, T, seed):
    from vlg_b200 import api
    gen = torch.Generator().manual_seed(seed)
    w = {"W1": torch.randn(K, 128, 2, generator=gen) * 0.7, "b1": torch.randn(K, 128, generator=gen) * 0.1,
         "W2": torch.randn(K, 128, 128, generator=gen) / 128 ** 0.5, "b2": torch.randn(K, 128, generator=gen) * 0.1,
         "W3": torch.randn(K, 50, 128, generator=gen) / 128 ** 0.5, "b3": torch.randn(K, 50, generator=gen) * 0.1}
    a = torch.rand(N, 2, generator=gen) * 6 - 3
    b = torch.rand(N, 2, generator=gen) * 6 - 3
    omega = 0.1 * torch.randn(N, n_poly + 1, 2, generator=gen)
    basis = api.construct_nullspace_basis(n_poly)[0]
    return w, a, b, omega, basis


@gpu
@pytest.mark.parametrize("prec", ["fp32", "f16x3f", "f16"])
def test_gradients_are_deterministic(vlg, prec):
    """Bit-identical gradients for a repeated launch, for the curve list split into two launches (curve_id0),
    and for a config-5-shaped case (K = 64, n_poly = 8, T = 256: several curves per window) regrouped."""
    g, model, dec, t, M, _ = _case(vlg, "synth_np4_T130", prec)
    N = model.omega.shape[0]
    r1 = energy_grad(vlg, model, dec, t, M, prec, seed=7)
    r2 = energy_grad(vlg, model, dec, t, M, prec, seed=7)
    for x, y in zip(r1[:4], r2[:4]):
        assert torch.equal(x, y)
    k = 2
    parts = []
    for lo, hi in ((0, k), (k, N)):
        m = vlg.GeodesicSplineBatch(model.a[lo:hi], model.b[lo:hi], model.basis, model.omega[lo:hi], model.n_poly)
        parts.append(energy_grad(vlg, m, dec, t, M, prec, seed=7, curve_id0=lo))
    for i in range(4):
        assert torch.equal(torch.cat([p[i] for p in parts]), r1[i])

    N5, K5, np5, T5 = 40, 64, 8, 256
    w, a, b, omega, basis = _random_case(N5, K5, np5, T5, 3)
    dec5 = vlg.DecoderEnsemble.from_arrays(*[w[k] for k in Hh.DEC_KEYS], "cuda")
    t5 = torch.linspace(0, 1, T5, device="cuda")
    full = vlg.GeodesicSplineBatch(a.cuda(), b.cuda(), basis.cuda(), omega.cuda(), np5)
    ref = energy_grad(vlg, full, dec5, t5, 2, prec, seed=11)
    assert ref[4] == 0
    for cut in (19, 33):
        parts = []
        for lo, hi in ((0, cut), (cut, N5)):
            m = vlg.GeodesicSplineBatch(full.a[lo:hi], full.b[lo:hi], full.basis, full.omega[lo:hi], np5)
            parts.append(energy_grad(vlg, m, dec5, t5, 2, prec, seed=11, curve_id0=lo))
        for i in range(4):
            assert torch.equal(torch.cat([p[i] for p in parts]), ref[i]), (cut, i)


@gpu
@pytest.mark.parametrize("prec", ["fp32", "f16x3f"])
def test_decoder_base_gives_the_per_set_bits(vlg, prec):
    """Two weight sets packed into one buffer, one launch with decoder_base == one launch per set."""
    g, model, dec, t, M, _ = _case(vlg, "synth_np4_T130", prec)
    K, N = int(g["K"]), model.omega.shape[0]
    arrs0 = Hh.decoder_arrays(g)
    arrs1 = {k: (v * 0.9 if k.startswith("W") else v) for k, v in arrs0.items()}
    both = vlg.DecoderEnsemble.from_arrays(*[np.concatenate([arrs0[k], arrs1[k]]) for k in Hh.DEC_KEYS], "cuda")
    sets = [vlg.DecoderEnsemble.from_arrays(*[arr[k] for k in Hh.DEC_KEYS], "cuda") for arr in (arrs0, arrs1)]
    cut = 2
    base = torch.tensor([0] * cut + [K] * (N - cut), dtype=torch.int32, device="cuda")
    active = vlg.DecoderEnsemble(both.packed, both.K, both.X, k_active=K)
    one = energy_grad(vlg, model, active, t, M, prec, seed=5, decoder_base=base)
    assert one[4] == 0
    for (lo, hi), s in zip(((0, cut), (cut, N)), sets):
        m = vlg.GeodesicSplineBatch(model.a[lo:hi], model.b[lo:hi], model.basis, model.omega[lo:hi], model.n_poly)
        part = energy_grad(vlg, m, s, t, M, prec, seed=5, curve_id0=lo)
        for i in range(4):
            assert torch.equal(part[i], one[i][lo:hi]), (lo, i)


@gpu
@pytest.mark.parametrize("prec", PRECISIONS)
def test_gradient_launch_writes_only_its_outputs(vlg, prec):
    """Inputs bit-unchanged; guard bands around energy and the three gradient buffers untouched."""
    g, model, dec, t, M, draws = _case(vlg, "synth_np8_T256", prec)
    N, Kb = model.omega.shape[0], model.omega.shape[1]
    before = [x.clone() for x in (model.omega, model.a, model.b, model.basis, t)]
    GB = 257
    shapes = [(N,), (N, Kb, 2), (N, 2), (N, 2)]
    bufs = [torch.full((2 * GB + int(np.prod(s)),), 12345.0, device="cuda") for s in shapes]
    outs = tuple(buf[GB:GB + int(np.prod(s))].view(s) for buf, s in zip(bufs, shapes))
    flags = energy_grad(vlg, model, dec, t, M, prec, draws, outs=outs)[4]
    assert flags == 0
    for x, y in zip(before, (model.omega, model.a, model.b, model.basis, t)):
        assert torch.equal(x, y)
    for buf in bufs:
        assert bool((buf[:GB] == 12345.0).all()) and bool((buf[-GB:] == 12345.0).all())
    for o in outs:
        assert bool(torch.isfinite(o).all())


@gpu
@pytest.mark.parametrize("prec", ["fp32", "tf32", "f16", "f16x3"])
def test_gradient_status_word_reports_bad_draws_and_overflow(vlg, prec):
    g, model, dec, t, _, _ = _case(vlg, "synth_np4_T130", prec)
    N, T, K, M = model.omega.shape[0], 130, 4, 2
    assert energy_grad(vlg, model, dec, t, M, prec)[4] == 0
    bad = torch.full((N, 1, M, 2, T - 1), 200, dtype=torch.uint8, device="cuda")
    E, gom, ga, gb, flags = energy_grad(vlg, model, dec, t, M, prec, bad)
    assert flags & 1 and all(bool(torch.isfinite(x).all()) for x in (E, gom, ga, gb))   # clamped, memory-safe
    # decoders whose hidden activations exceed the fp16 range
    arrs = {k: v.copy() for k, v in Hh.decoder_arrays(g).items()}
    arrs["W2"] = arrs["W2"] * 3.0e4
    big = vlg.DecoderEnsemble.from_arrays(*[arrs[k] for k in Hh.DEC_KEYS], "cuda")[:K]
    flags = energy_grad(vlg, model, big, t, M, prec)[4]
    if prec in ("f16", "f16x3"):
        assert flags & 2
        m = make_model(vlg, g)
        m.omega.requires_grad_(True)
        with pytest.raises(vlg.VlgError, match="fp16 range"):
            vlg.compute_energy_mc(m, big, t, M=M, precision=prec)
    else:
        assert flags == 0


@gpu
def test_spline_points_backward_matches_fp64_autograd(vlg):
    from oracle import torch_port as TP
    g = Hh.load("synth_np8_T256")
    n_poly, T = int(g["n_poly"]), int(g["T"])
    model = make_model(vlg, g)
    for x in (model.omega, model.a, model.b):
        x.requires_grad_(True)
    t = torch.linspace(0, 1, T, device="cuda")
    w = torch.randn(T, model.omega.shape[0], 2, generator=torch.Generator().manual_seed(0))

    def grads():
        for x in (model.omega, model.a, model.b):
            x.grad = None
        (model(t) * w.cuda()).sum().backward()
        return [x.grad.clone() for x in (model.omega, model.a, model.b)]

    r1, r2 = grads(), grads()
    for x, y in zip(r1, r2):
        assert torch.equal(x, y)
    a = torch.tensor(g["a"], dtype=torch.float64, requires_grad=True)
    b = torch.tensor(g["b"], dtype=torch.float64, requires_grad=True)
    sb = TP.SplineBatch(a, b, torch.tensor(g["basis"], dtype=torch.float64),
                        torch.tensor(g["omega_init"], dtype=torch.float64), n_poly)
    (sb(torch.tensor(Hh.tgrid(T), dtype=torch.float64)) * w.double()).sum().backward()
    for x, ref in zip(r1, (sb.omega.grad, a.grad, b.grad)):
        assert Hh.relerr(x.cpu().numpy(), ref.numpy()) < 1e-6


@gpu
def test_untracked_gradients_are_refused(vlg):
    g, model, dec, t, M, draws = _case(vlg, "synth_np4_T130", "fp32")
    model.omega.requires_grad_(True)
    model.basis.requires_grad_(True)
    with pytest.raises(vlg.VlgError, match="basis"):
        vlg.compute_energy_mc(model, dec, t, M, draws=draws.numpy())
    with pytest.raises(vlg.VlgError, match="basis"):
        model(t)
    model.basis.requires_grad_(False)
    with pytest.raises(vlg.VlgError, match="t_vals"):
        vlg.compute_energy_mc(model, dec, t.clone().requires_grad_(True), M, draws=draws.numpy())
    with pytest.raises(vlg.VlgError, match="return_length"):
        vlg.compute_energy_mc(model, dec, t, M, draws=draws.numpy(), return_length=True)
    E = vlg.compute_energy_mc(model, dec, t, M, draws=draws.numpy())
    (go,) = torch.autograd.grad(E.sum(), model.omega, create_graph=True)
    with pytest.raises(RuntimeError):
        go.sum().backward()
    z = model(t)
    (gz,) = torch.autograd.grad(z.sum(), model.omega, create_graph=True)
    with pytest.raises(RuntimeError):
        gz.sum().backward()
    # no grad wanted: the forward-only launch, the energy carries no grad_fn
    with torch.no_grad():
        assert vlg.compute_energy_mc(model, dec, t, M, draws=draws.numpy()).grad_fn is None
