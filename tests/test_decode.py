"""Decoder ensemble as a differentiable op: vlg_decode / vlg_decode_backward, DecoderEnsemble.__call__ and its
autograd Function, against the fp64 oracle and against the step kernels' own energy and gradient."""
import ctypes
import re
import warnings
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import geodesic_oracle as O
from tests import helpers as Hh

ROOT = Path(__file__).resolve().parent.parent
PRECISIONS = ["fp32", "f16x3", "f16x3f", "f16", "tf32"]
# Outputs, relative to the largest |x| (helpers.relerr).  Targets; measured maxima over the cases of
# test_outputs_and_input_gradient_match_fp64_oracle are recorded in DESIGN.md §4.6.
X_TOL = {"fp32": 1e-6, "f16x3": 1e-5, "f16x3f": 1e-5, "f16": 5e-3, "tf32": 5e-3}
# dz for random dx: the bounds of the step kernels' gradients (test_energy_grad.GRAD_TOL), on the points that lie
# away from every ReLU kink (KINK).  A pre-activation within rounding distance of 0 may take the other side of the
# kink in any fp32 evaluation; the gradient jumps there, by about as much as dz itself.  With 11-bit F2 operands
# (f16, tf32) the layer-2 masks flip within ~1e-3 of a kink, which excludes nearly every point of a 10-decoder
# ensemble (2560 pre-activations per point); their dz bound is the measured one (8.1e-2 before the margin).
GRAD_TOL = {"fp32": 2e-5, "f16x3": 2e-4, "f16x3f": 5e-3, "f16": 1.5e-1, "tf32": 1.5e-1}
KINK = 1e-5   # |pre-activation| below KINK x (the sum of the magnitudes of its terms), any decoder: excluded from dz
ERR_INVALID, ERR_UNSUPPORTED, ERR_WORKSPACE = -1, -2, -5
FAKE = 0x1000   # a non-null pointer: the argument checks run before any CUDA call and never dereference it


# ------------------------------------------------------------------ CPU ------------------------------------------

def test_header_declares_and_library_exports_the_decode_entries(built_lib):
    text = re.sub(r"/\*.*?\*/", "", (ROOT / "include" / "vlg.h").read_text(), flags=re.S)
    assert "vlg_decode(" in text and "vlg_decode_backward(" in text
    assert re.search(r"#define VLG_DECODE_WORKSPACE_BYTES 256\b", text)
    lib = ctypes.CDLL(str(built_lib))
    assert hasattr(lib, "vlg_decode") and hasattr(lib, "vlg_decode_backward")
    from vlg_b200 import _lib
    assert {"vlg_decode", "vlg_decode_backward"} <= set(_lib.SIGNATURES)


def test_decode_entries_reject_bad_arguments_before_any_device_call(built_lib):
    from vlg_b200 import _lib
    lib = _lib.load()

    def fwd(packed=FAKE, K=10, X=50, Ka=10, P=100, z=FAKE, x=FAKE, prec=4, ws=FAKE, wsb=256):
        return lib.vlg_decode(packed, K, X, Ka, P, z, x, prec, ws, wsb, None)

    def bwd(packed=FAKE, K=10, X=50, Ka=10, P=100, z=FAKE, dx=FAKE, dz=FAKE, prec=4, ws=FAKE, wsb=256):
        return lib.vlg_decode_backward(packed, K, X, Ka, P, z, dx, dz, prec, ws, wsb, None)

    for call, ptrs in ((fwd, ("packed", "z", "x", "ws")), (bwd, ("packed", "z", "dx", "dz", "ws"))):
        for name in ptrs:
            assert call(**{name: None}) == ERR_INVALID, name
        assert call(P=0) == ERR_INVALID and call(P=-5) == ERR_INVALID
        assert call(Ka=0) == ERR_INVALID and call(Ka=11) == ERR_INVALID
        assert call(prec=-1) == ERR_INVALID and call(prec=5) == ERR_INVALID
        assert call(X=53) == ERR_INVALID and call(K=255, Ka=1) == ERR_INVALID
        assert call(K=200, Ka=129, prec=2) == ERR_UNSUPPORTED
        assert call(K=200, Ka=129, prec=1, wsb=255) == ERR_UNSUPPORTED
        assert call(wsb=255) == ERR_WORKSPACE
        assert call(K=200, Ka=129, prec=0, wsb=0) == ERR_WORKSPACE


def test_decoder_call_refuses_cpu_tensors(built_lib):
    import vlg_b200
    ens = vlg_b200.DecoderEnsemble(torch.empty(0, dtype=torch.uint8), 10, 50)
    with pytest.raises(vlg_b200.VlgError, match="CUDA"):
        ens(torch.zeros(4, 2))


# ------------------------------------------------------------------ GPU ------------------------------------------

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def vlg(built_lib):
    import vlg_b200
    assert torch.cuda.is_available(), "GPU tests need a B200"
    return vlg_b200


def random_arrays(K, X, seed):
    """K decoders with torch.nn.Linear's default initialisation (uniform, bound 1/sqrt(fan_in))."""
    g = np.random.default_rng(seed)
    u = lambda shape, fan_in: g.uniform(-1, 1, shape) / np.sqrt(fan_in)
    return {"W1": u((K, 128, 2), 2), "b1": u((K, 128), 2), "W2": u((K, 128, 128), 128), "b2": u((K, 128), 128),
            "W3": u((K, X, 128), 128), "b3": u((K, X), 128)}


def seed12_arrays():
    return Hh.decoder_arrays(Hh.load("evae_seed12_decoders"))


def latent_box():
    grid = Hh.load("std_field_seed12")["grid"]
    return grid.min(0), grid.max(0)


def box_grid(n):
    lo, hi = latent_box()
    gx, gy = np.meshgrid(np.linspace(lo[0], hi[0], n), np.linspace(lo[1], hi[1], n), indexing="ij")
    return np.stack([gx.ravel(), gy.ravel()], 1).astype(np.float32)


def box_points(P, seed):
    lo, hi = latent_box()
    return np.random.default_rng(seed).uniform(lo, hi, (P, 2)).astype(np.float32)


def golden_curve_points():
    pts = []
    for tag in ("ens_seed12_euclid", "ens_seed12_entropy", "ens_seed12_cov_k3", "ens_seed12_long"):
        g = Hh.load(tag)
        T, n_poly = int(g["T"]), int(g["n_poly"])
        z = O.spline_points(g["a"].astype(np.float64), g["b"].astype(np.float64), g["omega_init"].astype(np.float64),
                            g["basis"].astype(np.float64), Hh.tgrid(T).astype(np.float64), n_poly)
        pts.append(z.reshape(-1, 2))
    return np.concatenate(pts).astype(np.float32)


def ensemble(vlg, arrs):
    return vlg.DecoderEnsemble.from_arrays(*[np.asarray(arrs[k], dtype=np.float32) for k in Hh.DEC_KEYS], "cuda")


def oracle(arrs, K, z, dx=None):
    """fp64 outputs [K,P,X], dz [P,2] = sum_k W1^T (m1 . W2^T (m2 . W3^T dx[k])) for dx [K,P,X], and the points
    away from every ReLU kink (KINK) [P] bool."""
    decs = Hh.decoder_list({k: np.asarray(v, dtype=np.float32) for k, v in arrs.items()}, K, np.float64)
    z = np.asarray(z, dtype=np.float64)
    xs, dz, keep = [], np.zeros_like(z), np.ones(z.shape[0], dtype=bool)
    for k, d in enumerate(decs):
        p1, p2, x = O.decoder_hidden(d, z)
        xs.append(x)
        s1 = np.abs(z) @ np.abs(d["W1"]).T + np.abs(d["b1"])
        s2 = np.maximum(p1, 0) @ np.abs(d["W2"]).T + np.abs(d["b2"])
        keep &= (np.abs(p1) >= KINK * s1).all(1) & (np.abs(p2) >= KINK * s2).all(1)
        if dx is not None:
            g2 = (np.asarray(dx[k], dtype=np.float64) @ d["W3"]) * (p2 > 0)
            dz += ((g2 @ d["W2"]) * (p1 > 0)) @ d["W1"]
    return np.stack(xs), dz, keep


def decode(ens, z, prec, dx=None):
    """(x, status) or, with dx, (dz, status) through the ops, without the Python-side status check."""
    from vlg_b200 import api, ops
    z = z.contiguous()
    code = api._resolve_precision(prec, ens, 1)
    ws = torch.empty(ops.DECODE_WORKSPACE_BYTES, dtype=torch.uint8, device="cuda")
    if dx is None:
        x = torch.empty((len(ens), z.shape[0], ens.X), device="cuda")
        ops.decode(ens.packed, ens.K, ens.X, len(ens), z, x, code, ws)
        return x, ops.workspace_status(ws)
    dz = torch.empty((z.shape[0], 2), device="cuda")
    ops.decode_backward(ens.packed, ens.K, ens.X, len(ens), z, dx.contiguous(), dz, code, ws)
    return dz, ops.workspace_status(ws)


CASES = {
    "seed12_grid": lambda: (seed12_arrays(), 10, box_grid(200)),
    "seed12_curves": lambda: (seed12_arrays(), 10, golden_curve_points()),
    "single_vae": lambda: (Hh.decoder_arrays(Hh.load("single_seed123")), 1, box_points(5000, 1)),
    "random_k64": lambda: (random_arrays(64, 50, 64), 64, box_points(3000, 2)),
    "random_k128": lambda: (random_arrays(128, 50, 128), 128, box_points(1000, 3)),
    "random_k129": lambda: (random_arrays(129, 50, 129), 129, box_points(1000, 4)),
    "random_x52": lambda: (random_arrays(10, 52, 52), 10, box_points(3000, 5)),
}


@gpu
@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("case", list(CASES))
def test_outputs_and_input_gradient_match_fp64_oracle(vlg, case, prec):
    arrs, K, z = CASES[case]()
    ens = ensemble(vlg, arrs)[:K]
    dx = np.random.default_rng(7).standard_normal((K, z.shape[0], ens.X)).astype(np.float32)
    x_ref, dz_ref, keep = oracle(arrs, K, z, dx)
    zt = torch.tensor(z, device="cuda", requires_grad=True)
    fallback = prec != "fp32" and (K > 128 or (K == 1 and prec in ("f16", "tf32")))
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        x = ens(zt, precision=prec)
        x.backward(torch.tensor(dx, device="cuda"))
    assert any("fp32 kernel" in str(w.message) for w in caught) == fallback
    ex = Hh.relerr(x.detach().cpu().numpy(), x_ref)
    ez = Hh.relerr(zt.grad.cpu().numpy()[keep], dz_ref[keep])
    print(f"{case} {prec}: x {ex:.2e} dz {ez:.2e} on {keep.mean():.0%} of the points")
    assert ex <= X_TOL[prec]
    assert ez <= GRAD_TOL[prec]


@gpu
@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("P", [1, 127, 128, 129, 1000])
def test_edge_sizes(vlg, P, prec):
    arrs = seed12_arrays()
    ens = ensemble(vlg, arrs)
    z = box_points(P, P)
    dx = np.random.default_rng(P).standard_normal((10, P, 50)).astype(np.float32)
    x_ref, dz_ref, keep = oracle(arrs, 10, z, dx)
    zt = torch.tensor(z, device="cuda")
    x, st = decode(ens, zt, prec)
    dz, st2 = decode(ens, zt, prec, torch.tensor(dx, device="cuda"))
    assert st == 0 and st2 == 0
    assert Hh.relerr(x.cpu().numpy(), x_ref) <= X_TOL[prec]
    if keep.any():
        assert Hh.relerr(dz.cpu().numpy()[keep], dz_ref[keep]) <= GRAD_TOL[prec]


@gpu
@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("tag", ["ens_seed12_euclid", "ens_seed12_entropy", "ens_seed12_cov_k3", "ens_seed12_long"])
def test_plain_torch_energy_matches_the_step_kernel(vlg, tag, prec):
    """The reference's compute_energy_mc (src/optimize.py:38-75) in plain torch on decoders(model(t_vals)), with
    autograd through _SplinePoints and _Decode, against vlg_b200.compute_energy_mc on the same draws."""
    g = Hh.load(tag)
    K, T, M = int(g["K"]), int(g["T"]), int(g["M"])
    N = g["a"].shape[0]
    draws = Hh.regen_draws(g)[0]                   # [M,2,T-1,N]
    ens = ensemble(vlg, Hh.decoder_arrays(g))[:K]
    t = torch.linspace(0, 1, T, device="cuda")

    def model():
        m = vlg.GeodesicSplineBatch(torch.tensor(g["a"], device="cuda"), torch.tensor(g["b"], device="cuda"),
                                    torch.tensor(g["basis"], device="cuda"), torch.tensor(g["omega_init"], device="cuda"),
                                    int(g["n_poly"]))
        for p in (m.omega, m.a, m.b):
            p.requires_grad_(True)
        return m

    m1 = model()
    X = ens(m1(t), precision=prec)                 # [K,T,N,X]
    d = torch.as_tensor(draws, device="cuda").long()
    it, ib = torch.arange(T - 1, device="cuda")[:, None], torch.arange(N, device="cuda")[None, :]
    E = sum(((X[d[m, 1], it + 1, ib] - X[d[m, 0], it, ib]) ** 2).sum(-1).sum(0) for m in range(M)) / M
    E.sum().backward()

    m2 = model()
    E2 = vlg.compute_energy_mc(m2, ens, t, M, draws=draws, precision=prec)
    E2.sum().backward()
    e_tol = 1e-5 if prec in ("fp32", "f16x3", "f16x3f") else GRAD_TOL[prec]
    errs = [Hh.relerr(E.detach().cpu().numpy(), E2.detach().cpu().numpy())]
    errs += [Hh.relerr(getattr(m1, k).grad.cpu().numpy(), getattr(m2, k).grad.cpu().numpy()) for k in ("omega", "a", "b")]
    print(f"{tag} {prec}: E {errs[0]:.2e} omega {errs[1]:.2e} a {errs[2]:.2e} b {errs[3]:.2e}")
    assert errs[0] <= e_tol
    assert max(errs[1:]) <= GRAD_TOL[prec]


@gpu
@pytest.mark.parametrize("prec", PRECISIONS)
def test_decode_is_deterministic_per_point(vlg, prec):
    ens = ensemble(vlg, seed12_arrays())
    P = 3001
    z = torch.tensor(box_points(P, 11), device="cuda")
    dx = torch.randn((10, P, 50), device="cuda", generator=torch.Generator("cuda").manual_seed(3))
    x0, _ = decode(ens, z, prec)
    dz0, _ = decode(ens, z, prec, dx)
    for _ in range(2):
        assert torch.equal(decode(ens, z, prec)[0], x0)
        assert torch.equal(decode(ens, z, prec, dx)[0], dz0)
    perm = torch.randperm(P, device="cuda", generator=torch.Generator("cuda").manual_seed(5))
    assert torch.equal(decode(ens, z[perm], prec)[0], x0[:, perm])
    assert torch.equal(decode(ens, z[perm], prec, dx[:, perm])[0], dz0[perm])
    s = 1234
    xa, xb = decode(ens, z[:s], prec)[0], decode(ens, z[s:], prec)[0]
    assert torch.equal(torch.cat([xa, xb], 1), x0)
    da, db = decode(ens, z[:s], prec, dx[:, :s])[0], decode(ens, z[s:], prec, dx[:, s:])[0]
    assert torch.equal(torch.cat([da, db]), dz0)


@gpu
@pytest.mark.parametrize("prec", PRECISIONS)
def test_backward_scales_exactly_with_dx(vlg, prec):
    ens = ensemble(vlg, seed12_arrays())
    P = 1000
    z = torch.tensor(box_points(P, 12), device="cuda")
    dx = torch.randn((10, P, 50), device="cuda", generator=torch.Generator("cuda").manual_seed(4))
    zero = torch.arange(0, P, 7, device="cuda")
    dx[:, zero] = 0
    dz, st = decode(ens, z, prec, dx)
    assert st == 0
    assert torch.equal(dz[zero], torch.zeros_like(dz[zero]))
    assert bool((dz.abs().sum(1) > 0).sum() == P - zero.numel())
    for e in (-30, -10, 10, 30):
        assert torch.equal(decode(ens, z, prec, dx * 2.0 ** e)[0], dz * 2.0 ** e), e


@gpu
@pytest.mark.parametrize("prec", PRECISIONS)
def test_decode_writes_only_inside_its_buffers(vlg, prec):
    from vlg_b200 import api, ops
    ens = ensemble(vlg, seed12_arrays())
    P, pad, S = 300, 4096, -12345.0
    code = api._resolve_precision(prec, ens, 1)
    z = torch.tensor(box_points(P, 13), device="cuda")
    ws = torch.empty(256, dtype=torch.uint8, device="cuda")
    n = 10 * P * 50
    xbuf = torch.full((n + 2 * pad,), S, device="cuda")
    ops.decode(ens.packed, ens.K, ens.X, 10, z, xbuf[pad:pad + n].view(10, P, 50), code, ws)
    dzbuf = torch.full((2 * P + 2 * pad,), S, device="cuda")
    dx = torch.randn((10, P, 50), device="cuda")
    ops.decode_backward(ens.packed, ens.K, ens.X, 10, z, dx, dzbuf[pad:pad + 2 * P].view(P, 2), code, ws)
    torch.cuda.synchronize()
    for buf, m in ((xbuf, n), (dzbuf, 2 * P)):
        assert bool((buf[:pad] == S).all()) and bool((buf[pad + m:] == S).all())
        assert not bool((buf[pad:pad + m] == S).any())


@gpu
@pytest.mark.parametrize("prec", PRECISIONS)
def test_decode_status_word(vlg, prec):
    from vlg_b200 import ops
    ens = ensemble(vlg, seed12_arrays())
    z = torch.tensor(box_points(200, 14), device="cuda")
    z[77, 0] = float("inf")
    _, st = decode(ens, z, prec)
    assert st & ops.STATUS_NONFINITE
    _, st = decode(ens, z, prec, torch.randn((10, 200, 50), device="cuda"))
    assert st & ops.STATUS_NONFINITE
    with pytest.raises(vlg.VlgError, match="non-finite"):
        ens(z, precision=prec)
    x = ens(z, precision=prec, check=False)
    assert x.shape == (10, 200, 50)
    zok = torch.tensor(box_points(200, 15), device="cuda")
    wrong = vlg.DecoderEnsemble(ens.packed, ens.K, 48)
    _, st = decode(wrong, zok, prec)
    assert st == ops.STATUS_BAD_PACKED
    with pytest.raises(vlg.VlgError, match="does not match its K / X"):
        wrong(zok, precision=prec)


@gpu
def test_decoder_call_shapes_and_refusals(vlg):
    ens = ensemble(vlg, seed12_arrays())
    z = torch.tensor(box_points(60, 16), device="cuda").reshape(3, 20, 2)
    x = ens(z)
    assert x.shape == (10, 3, 20, 50) and x.dtype == torch.float32 and x.grad_fn is None
    assert torch.equal(ens[:4](z), x[:4])
    assert torch.equal(ens(z.double()), x)
    with pytest.raises(vlg.VlgError, match=r"\[\.\.\., 2\]"):
        ens(torch.zeros(5, 3, device="cuda"))
    with pytest.raises(vlg.VlgError, match="CUDA"):
        ens(z.cpu())
    zg = z.double().requires_grad_(True)
    y = ens(zg)
    (gz,) = torch.autograd.grad(y.sum(), zg)
    assert gz.dtype == torch.float64 and gz.shape == zg.shape
    with pytest.raises(vlg.VlgError, match="double backward"):
        torch.autograd.grad(ens(zg).sum(), zg, create_graph=True)
    with torch.no_grad():
        assert ens(zg).grad_fn is None


@gpu
def test_decode_indexes_beyond_2_to_the_31(vlg):
    """K_active * P * X > 2^31 (about 9 GB per tensor): the last tile's rows against the oracle."""
    arrs = seed12_arrays()
    ens = ensemble(vlg, arrs)
    P = 4_500_000 + 77
    assert 10 * P * 50 > 2 ** 31
    z = torch.tensor(box_points(P, 17), device="cuda")
    tail = slice(P - 205, P)
    x, st = decode(ens, z, "f16x3")
    assert st == 0
    zt = z[tail].cpu().numpy()
    dxt = np.random.default_rng(8).standard_normal((10, zt.shape[0], 50)).astype(np.float32)
    x_ref, dz_ref, keep = oracle(arrs, 10, zt, dxt)
    assert Hh.relerr(x[:, tail].cpu().numpy(), x_ref) <= X_TOL["f16x3"]
    dx = torch.zeros_like(x)
    del x
    dx[:, tail] = torch.tensor(dxt, device="cuda")
    dz, st = decode(ens, z, "f16x3", dx)
    assert st == 0
    assert Hh.relerr(dz[tail].cpu().numpy()[keep], dz_ref[keep]) <= GRAD_TOL["f16x3"]
    assert bool((dz[:P - 205] == 0).all())
