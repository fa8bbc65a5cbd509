"""Every launch plan of the step kernels against a sparse fp64 reference.

The tensor-core step kernel picks its plan from (T, K, M) on the host (tc_plan, csrc/vlg_tc.cu): one window per
curve, several windows per curve, the left-end outputs in shared memory or in the L2 workspace, G whole curves per
window, and one curve per window with per-curve weight sets (decoder_base).  The window indexing and the home of the
end-point outputs differ between them, so each plan is checked here on its own: the energy, the poly-line length,
dE/domega, dE/da, dE/db and three Adam steps, in every precision, with explicit and with counter-based draws.

The reference evaluates each decoder only on the points that drew it (fp64 torch, autograd for the gradients), so it
stays cheap at T = 2000 with up to 254 decoders.  A CPU test pins it to the dense oracles."""
import functools
import warnings

import numpy as np
import pytest
import torch

from oracle import geodesic_oracle as O
from oracle import torch_port as TP
from tests import helpers as Hh

F64 = torch.float64
PRECISIONS = ["fp32", "f16x3", "f16x3f", "f16", "tf32"]
ELEVEN_BIT = ("f16", "tf32")
LR, BETA1, PENALTY = 1e-3, 0.9, 1000.0
STEPS = 3

# Bounds per arithmetic, set before the first run.  Energy and length: relative error per curve (the 11-bit modes:
# of sqrt(energy), the geodesic length, and of the poly-line length).  Gradients: per curve, the largest error of
# dE/domega, dE/da and dE/db relative to the largest entry of the three.
TOL = {"fp32": dict(E=5e-6, L=5e-6, G=2e-5),
       "f16x3": dict(E=1e-5, L=1e-5, G=2e-4),
       "f16x3f": dict(E=1e-5, L=1e-5, G=5e-3),
       "f16": dict(E=1e-3, L=1e-3, G=6e-2),
       "tf32": dict(E=1e-3, L=1e-3, G=6e-2)}
# The 11-bit modes on default-init (nn.Linear) decoders at K >= 64: 3x the largest error measured on one B200
# (sqrt(E) 9.5e-5, length 9.6e-5, gradients 8.6e-3 at K = 128, T = 3).
TOL_11BIT_DEFAULT_INIT = dict(E=3e-4, L=3e-4, G=2.6e-2)
# The 11-bit modes with fewer than 10 real decoders: a quarter of the K = 4 pairs subtract two outputs of one decoder at
# neighbouring points, the cancellation the single-decoder energy suffers from (the package runs K = 1 on the fp32
# kernel for this reason).  One B200 measured sqrt(E) 1.0e-3 and length 1.08e-3 on K = 4, M = 1 with f16 and with
# tf32 alike (operand rounding, not a code path); the bound is 3x that.  With 10 or more the largest is 3.8e-4.
TOL_11BIT_FEW_DECODERS = dict(E=3.3e-3, L=3.3e-3, G=6e-2)
# Three free-running Adam steps: per-step energies (relative, per curve) and omega (absolute).  Adam's first steps
# move each coefficient by ~lr whatever the gradient's size, so an 11-bit gradient operand (f16x3f's backward, f16,
# tf32) that flips the sign of a near-zero component costs up to 2 lr per step.
TRACE_TOL = {"fp32": 1e-5, "f16x3": 1e-4, "f16x3f": 1e-3, "f16": 5e-3, "tf32": 5e-3}
OMEGA_TOL = {"fp32": 5e-6, "f16x3": 2e-5, "f16x3f": 0.25 * STEPS * LR + 1e-6, "f16": 0.25 * STEPS * LR + 1e-6,
             "tf32": 0.25 * STEPS * LR + 1e-6}


# ------------------------------------------------------------------ decoders and cases --------------------------

@functools.lru_cache(maxsize=None)
def real_decoders():
    """The 60 trained eVAE decoders of the six seeds of the CoV study (10 each), as one dict of arrays."""
    g = np.load(Hh.GOLDEN / "evae_six_seeds.npz")
    out = {k: [] for k in Hh.DEC_KEYS}
    for s in (int(x) for x in g["seeds"]):
        for i in range(10):
            for name, layer in (("1", 0), ("2", 2), ("3", 4)):
                out["W" + name].append(g[f"s{s}/decoder.{i}.decoder_net.{layer}.weight"])
                out["b" + name].append(g[f"s{s}/decoder.{i}.decoder_net.{layer}.bias"])
    return {k: np.stack(v).astype(np.float32) for k, v in out.items()}


@functools.lru_cache(maxsize=None)
def default_init_decoders(K, seed=0):
    """K decoders 2 -> 128 -> 128 -> 50 with the default nn.Linear init (BASELINE config 5)."""
    import torch.nn as nn
    torch.manual_seed(seed)
    nets = [nn.Sequential(nn.Linear(2, 128), nn.ReLU(), nn.Linear(128, 128), nn.ReLU(), nn.Linear(128, 50))
            for _ in range(K)]
    W = {}
    for name, idx in (("1", 0), ("2", 2), ("3", 4)):
        W["W" + name] = torch.stack([n_[idx].weight.detach() for n_ in nets]).numpy()
        W["b" + name] = torch.stack([n_[idx].bias.detach() for n_ in nets]).numpy()
    return W


def decoder_arrays(K, X=50):
    """Real decoders for K <= 60, default init beyond.  X != 50: the real decoders' first X outputs, or two extra
    outputs for X = 52."""
    W = {k: v[:K] for k, v in real_decoders().items()} if K <= 60 else dict(default_init_decoders(K))
    if X < 50:
        W["W3"], W["b3"] = W["W3"][:, :X], W["b3"][:, :X]
    elif X > 50:
        rng = np.random.default_rng(X)
        W["W3"] = np.concatenate([W["W3"], (0.09 * rng.normal(size=(K, X - 50, 128))).astype(np.float32)], 1)
        W["b3"] = np.concatenate([W["b3"], (0.1 * rng.normal(size=(K, X - 50))).astype(np.float32)], 1)
    return {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in W.items()}


def nonuniform_grid(T, n_poly, seed=0):
    """Sorted fp32 grid with t[0] = 0, t[-1] = 1 and a point exactly on every knot j / n_poly."""
    rng = np.random.default_rng(seed)
    knots = np.arange(n_poly + 1, dtype=np.float64) / n_poly
    t = np.concatenate([knots, rng.uniform(0, 1, T - n_poly - 1)]).astype(np.float32)
    return np.sort(t)


#              N   T     K    M  n_poly  sets  grid
CASES = {
    # R1: shared-memory home, one window per curve
    "r1_T130_K4_M1": (3, 130, 4, 1, 4, 1, "uniform"),
    "r1_T40_K10_M2": (4, 40, 10, 2, 4, 1, "uniform"),
    # R2: shared-memory home, several windows per curve (T = 2001: the last window is short)
    "r2_T2000_K10_M2": (3, 2000, 10, 2, 4, 1, "uniform"),
    "r2_T2000_K10_M3": (3, 2000, 10, 3, 4, 1, "uniform"),
    "r2_T2001_K10_M2": (3, 2001, 10, 2, 4, 1, "uniform"),
    # R3: L2 home, one curve per window, several windows per curve; K = 64, M = 1: shared memory, W = 501
    "r3_T1000_K32_M2": (3, 1000, 32, 2, 4, 1, "uniform"),
    "r3_T2000_K60_M2": (3, 2000, 60, 2, 4, 1, "uniform"),
    "r3_T2000_K60_M3": (3, 2000, 60, 3, 4, 1, "uniform"),
    "r3_T2000_K64_M1": (3, 2000, 64, 1, 4, 1, "uniform"),
    # R4: L2 home, G whole curves per window (N = 23 at G = 7: the last group is partial; G = 8 with n_poly 8)
    "r4_T256_K60_M2_N23": (23, 256, 60, 2, 4, 1, "uniform"),
    "r4_T256_K16_M3": (8, 256, 16, 3, 4, 1, "uniform"),
    "r4_T96_K16_M1_np8": (10, 96, 16, 1, 8, 1, "uniform"),
    # R5: per-curve weight sets (decoder_base), one curve per window: L2 home at T = 1000, shared memory at 2000
    "r5_2x30_T1000": (4, 1000, 30, 2, 4, 2, "uniform"),
    "r5_6x10_T2000": (6, 2000, 10, 2, 4, 6, "uniform"),
    # limits: the tensor-core maximum K = 128 (T = 800: G = 2), one and two segments, M beyond the fp32 kernel's
    # four, K beyond the tensor-core kernel's 128 (falls back to the fp32 kernel), the fp32 kernel's K and M limits
    "lim_K128_T800": (3, 800, 128, 2, 4, 1, "uniform"),
    "lim_K128_T2": (3, 2, 128, 2, 4, 1, "uniform"),
    "lim_K128_T3": (3, 3, 128, 2, 4, 1, "uniform"),
    "lim_M5_T40": (3, 40, 10, 5, 4, 1, "uniform"),
    "lim_M64_T40": (2, 40, 10, 64, 4, 1, "uniform"),
    "lim_K129_T40": (3, 40, 129, 2, 4, 1, "uniform"),
    "lim_K254_M4_T40": (3, 40, 254, 4, 4, 1, "uniform"),
    # the kernels read t[] everywhere: a non-uniform grid with points on the knots
    "grid_nonuniform": (3, 300, 10, 2, 4, 1, "knots"),
}
FP32_MAX_M, TC_MAX_K = 4, 128


# forced plans (VLG_TC_XL2 / VLG_TC_G / VLG_TC_WINDOW): the same inputs through every admissible home and grouping
_SMEM, _L2 = {"VLG_TC_XL2": "0"}, {"VLG_TC_XL2": "1"}
FORCED = {
    "plan_T256_K16": ((17, 256, 16, 2, 4, 1, "uniform"),
                      [("smem", _SMEM)] + [(f"l2_G{g}", dict(_L2, VLG_TC_G=str(g))) for g in range(2, 9)]),
    "plan_T256_K60": ((17, 256, 60, 2, 4, 1, "uniform"),
                      [("smem", _SMEM)] + [(f"l2_G{g}", dict(_L2, VLG_TC_G=str(g))) for g in range(2, 9)]),
    "plan_T1000_K32": ((3, 1000, 32, 2, 4, 1, "uniform"),
                       [("smem_W251", dict(_SMEM, VLG_TC_WINDOW="4")), ("l2_W501", dict(_L2, VLG_TC_WINDOW="2"))]),
    "plan_T2000_K60": ((3, 2000, 60, 2, 4, 1, "uniform"),
                       [("smem_W287", dict(_SMEM, VLG_TC_WINDOW="7")), ("l2_W501", dict(_L2, VLG_TC_WINDOW="4"))]),
}


def shape(name):
    return CASES[name] if name in CASES else FORCED[name][0]


def regime(name):
    return name.split("_")[0]


def default_init(name):
    return shape(name)[2] * shape(name)[5] > 60


def effective_precision(name, prec):
    """What the package runs: more than 128 decoders fall back to the fp32 kernel."""
    return "fp32" if shape(name)[2] > TC_MAX_K else prec


def tolerances(name, prec):
    prec = effective_precision(name, prec)
    if prec in ELEVEN_BIT and default_init(name):
        return TOL_11BIT_DEFAULT_INIT
    if prec in ELEVEN_BIT and shape(name)[2] < 10:
        return TOL_11BIT_FEW_DECODERS
    return TOL[prec]


@functools.lru_cache(maxsize=None)
def case_inputs(name, X=50):
    """Host inputs of a case: spline batch (fp32), grid, decoder arrays, decoder_base, active decoders per curve."""
    from vlg_b200 import api
    N, T, K, M, n_poly, sets, grid = shape(name)
    rng = np.random.default_rng(sum(map(ord, name)))
    W = decoder_arrays(K * sets, X)
    base = None if sets == 1 else (np.arange(N) * sets // N * K).astype(np.int32)
    t = nonuniform_grid(T, n_poly) if grid == "knots" else Hh.tgrid(T)
    return dict(N=N, T=T, K=K, M=M, n_poly=n_poly, W=W, base=base, t=t,
                a=rng.uniform(-2, 2, (N, 2)).astype(np.float32), b=rng.uniform(-2, 2, (N, 2)).astype(np.float32),
                omega=(0.1 * rng.normal(size=(N, n_poly + 1, 2))).astype(np.float32),
                basis=api.construct_nullspace_basis(n_poly)[0].numpy())


SEED, CURVE_ID0 = 7, 3


@functools.lru_cache(maxsize=None)
def case_draws(name, mode, X=50):
    """Local decoder draws [S, M, 2, T-1, N] of STEPS steps: explicit (uniform random), or the counter-based
    stream the kernels form themselves (seed SEED, curve ids CURVE_ID0 ...)."""
    c = case_inputs(name, X)
    N, T, K, M = c["N"], c["T"], c["K"], c["M"]
    if mode == "explicit":
        return np.random.default_rng(11).integers(0, K, size=(STEPS, M, 2, T - 1, N))
    ids = CURVE_ID0 + np.arange(N)
    return np.stack([O.counter_draws(SEED, ids, s, T, M, K) for s in range(STEPS)])


# ------------------------------------------------------------------ the fp64 reference --------------------------

def fp64_nets(W):
    nets = [TP.make_decoder({k: v[i].astype(np.float64) for k, v in W.items()}).double()
            for i in range(W["W1"].shape[0])]
    for net in nets:
        net.requires_grad_(False)
    return nets


def sparse_reference(nets, a, b, omega, basis, t, n_poly, draws, base=None, penalty_w=0.0):
    """fp64 energy E = (1/M) sum ||x2 - x1||^2, length (1/M) sum ||x2 - x1||, and d(E + penalty_w ||z(t[-1]) - b||^2)
    with respect to omega, a and b (torch.autograd).  Each decoder runs only on the points that drew it.

    nets: fp64 decoders; draws [M, 2, T-1, N] local indices (curve n uses nets[base[n] + d]); t: the kernels' grid
    values (fp32 widened to fp64)."""
    ta = torch.tensor(np.asarray(a), dtype=F64, requires_grad=True)
    tb = torch.tensor(np.asarray(b), dtype=F64, requires_grad=True)
    sb = TP.SplineBatch(ta, tb, torch.tensor(np.asarray(basis), dtype=F64), torch.tensor(np.asarray(omega), dtype=F64),
                        n_poly)
    tt = torch.tensor(np.asarray(t), dtype=F64)
    z = sb(tt)                                                        # [T, N, 2]
    T, N = z.shape[0], z.shape[1]
    d = torch.as_tensor(np.asarray(draws), dtype=torch.int64)         # [M, 2, T-1, N]
    M = d.shape[0]
    if base is not None:
        d = d + torch.as_tensor(np.asarray(base), dtype=torch.int64)
    zz = torch.stack([z[:-1], z[1:]]).expand(M, 2, T - 1, N, 2)       # role 0: left points, role 1: right points
    x = z.new_zeros(M, 2, T - 1, N, nets[0][4].out_features)
    for k in torch.unique(d).tolist():
        sel = d == k
        x[sel] = nets[k](zz[sel])
    sq = ((x[:, 1] - x[:, 0]) ** 2).sum(-1)                           # [M, T-1, N]
    E = sq.sum((0, 1)) / M
    L = sq.detach().sqrt().sum((0, 1)) / M
    loss = E
    if penalty_w:
        loss = E + penalty_w * ((sb(tt[-1:])[0] - tb) ** 2).sum(-1)
    go, ga, gb = torch.autograd.grad(loss.sum(), (sb.omega, ta, tb))
    return dict(E=E.detach().numpy(), L=L.numpy(), gom=go.numpy(), ga=ga.numpy(), gb=gb.numpy())


def reference_adam(nets, c, draws, steps, step0=0):
    """steps of the reference loop (energy + end-point penalty, torch.optim.Adam) in fp64: energies [S, N], omega."""
    om = c["omega"].astype(np.float64)
    m, v = np.zeros_like(om), np.zeros_like(om)
    energies = []
    for s in range(steps):
        r = sparse_reference(nets, c["a"], c["b"], om, c["basis"], c["t"], c["n_poly"], draws[s], c["base"],
                             penalty_w=PENALTY)
        energies.append(r["E"])
        om, m, v = O.adam_update(om, m, v, r["gom"], step0 + s + 1, lr=LR)
    return np.stack(energies), om


@functools.lru_cache(maxsize=None)
def case_reference(name, mode, X=50):
    c = case_inputs(name, X)
    nets = fp64_nets(c["W"])
    d = case_draws(name, mode, X)
    r = sparse_reference(nets, c["a"], c["b"], c["omega"], c["basis"], c["t"], c["n_poly"], d[0], c["base"])
    r["trace"], r["omega_S"] = reference_adam(nets, c, d, STEPS)
    return r


# ------------------------------------------------------------------ CPU ------------------------------------------

@pytest.mark.parametrize("K", [3, 7])
def test_sparse_reference_matches_the_dense_oracles(K):
    """The sparse reference against O.energy_mc_grad (energy, dE/domega), oracle.torch_port autograd (dE/da,
    dE/db) and a dense numpy poly-line length, to 1e-12."""
    from vlg_b200 import api
    N, T, M, n_poly = 3, 37, 3, 8
    rng = np.random.default_rng(K)
    W = {k: v[:K].astype(np.float64) for k, v in Hh.load("evae_seed12_decoders").items() if k in Hh.DEC_KEYS}
    decs = Hh.decoder_list(W, K, np.float64)
    a, b = rng.uniform(-2, 2, (N, 2)), rng.uniform(-2, 2, (N, 2))
    om = 0.1 * rng.normal(size=(N, n_poly + 1, 2))
    basis = api.construct_nullspace_basis(n_poly)[0].numpy().astype(np.float64)
    t = Hh.tgrid(T, np.float64)
    draws = rng.integers(0, K, size=(M, 2, T - 1, N))
    nets = fp64_nets(W)
    r = sparse_reference(nets, a, b, om, basis, t, n_poly, draws)

    E, grad, _ = O.energy_mc_grad(a, b, om, basis, t, n_poly, decs, draws, penalty_w=0.0)
    assert Hh.relerr(r["E"], E) < 1e-12
    assert Hh.relerr(r["gom"], grad) < 1e-12

    ta = torch.tensor(a, requires_grad=True)
    tb = torch.tensor(b, requires_grad=True)
    sb = TP.SplineBatch(ta, tb, torch.tensor(basis), torch.tensor(om), n_poly)
    e = TP.energy_mc(sb, [TP.make_decoder(w).double() for w in decs], torch.tensor(t), M, torch.as_tensor(draws))
    e.sum().backward()
    assert Hh.relerr(r["ga"], ta.grad.numpy()) < 1e-12
    assert Hh.relerr(r["gb"], tb.grad.numpy()) < 1e-12
    assert Hh.relerr(r["gom"], sb.omega.grad.numpy()) < 1e-12

    z = O.spline_points(a, b, om, basis, t, n_poly).reshape(T * N, 2)
    X = np.stack([O.decoder_mean(dd, z).reshape(T, N, -1) for dd in decs])
    it, ib = np.arange(T - 1)[:, None], np.arange(N)[None, :]
    L = sum(np.linalg.norm(X[draws[m, 1], it + 1, ib] - X[draws[m, 0], it, ib], axis=-1).sum(0) for m in range(M)) / M
    assert Hh.relerr(r["L"], L) < 1e-12


def test_packed_decoders_accept_at_most_52_outputs(built_lib):
    from vlg_b200 import _lib
    lib = _lib.load()
    for X in (1, 3, 49, 50, 52):
        assert lib.vlg_packed_decoders_bytes(10, 128, X) > 0, X
    assert lib.vlg_packed_decoders_bytes(128, 128, 52) > 0
    for X in (0, 53, 64):
        assert lib.vlg_packed_decoders_bytes(128, 128, X) == 0, X


# ------------------------------------------------------------------ GPU helpers ----------------------------------

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def vlg(built_lib):
    import vlg_b200
    assert torch.cuda.is_available(), "GPU tests need a B200"
    return vlg_b200


class Run:
    """Device inputs of a case and the three launches under test."""

    def __init__(self, vlg, name, mode, X=50):
        self.vlg, self.name, self.mode = vlg, name, mode
        self.c = c = case_inputs(name, X)
        self.N, self.T, self.K, self.M, self.n_poly = c["N"], c["T"], c["K"], c["M"], c["n_poly"]
        self.packed = vlg.DecoderEnsemble.from_arrays(*[c["W"][k] for k in Hh.DEC_KEYS], "cuda")
        self.dec = vlg.DecoderEnsemble(self.packed.packed, self.packed.K, self.packed.X, k_active=self.K)
        self.base = None if c["base"] is None else torch.tensor(c["base"], device="cuda")
        self.t = torch.tensor(c["t"], device="cuda")
        self.draws = case_draws(name, mode, X) if mode == "explicit" else None
        self.seed, self.id0 = (0, 0) if mode == "explicit" else (SEED, CURVE_ID0)

    def model(self):
        c = self.c
        return self.vlg.GeodesicSplineBatch(*(torch.tensor(c[k], device="cuda") for k in ("a", "b", "basis", "omega")),
                                            self.n_poly)

    def code(self, prec):
        from vlg_b200 import api
        return api._resolve_precision(prec, self.dec, self.M)

    def _launch_args(self, model, prec):
        from vlg_b200 import api
        code = self.code(prec)
        ws = api._workspace(model, self.dec, self.T, self.M, code)
        d = None if self.draws is None else api._prep_draws(self.draws[0], self.N, 1, self.M, self.T, "cuda", self.K)
        return code, ws, d

    def grad(self, prec):
        """vlg_curve_energy_grad -> dict of host arrays E, gom, ga, gb and the status flags."""
        from vlg_b200 import ops
        m = self.model()
        code, ws, d = self._launch_args(m, prec)
        E, gom = torch.empty(self.N, device="cuda"), torch.empty_like(m.omega)
        ga, gb = torch.empty(self.N, 2, device="cuda"), torch.empty(self.N, 2, device="cuda")
        ops.curve_energy_grad(self.dec.packed, self.dec.K, self.dec.X, self.K, self.n_poly, self.M, m.a, m.b, m.omega,
                              m.basis, self.t, d, self.base, self.seed, self.id0, 0, E, gom, ga, gb, code, ws)
        flags = ops.workspace_status(ws)
        return dict(E_t=E, E=E.cpu().numpy(), gom=gom.cpu().numpy(), ga=ga.cpu().numpy(), gb=gb.cpu().numpy(),
                    flags=flags)

    def forward(self, prec):
        """vlg_curve_energy with the length -> dict E, L and the status flags."""
        from vlg_b200 import ops
        m = self.model()
        code, ws, d = self._launch_args(m, prec)
        E, L = torch.empty(self.N, device="cuda"), torch.empty(self.N, device="cuda")
        ops.curve_energy(self.dec.packed, self.dec.K, self.dec.X, self.K, self.n_poly, self.M, m.a, m.b, m.omega,
                         m.basis, self.t, d, self.base, self.seed, self.id0, 0, E, L, code, ws)
        return dict(E=E.cpu().numpy(), L=L.cpu().numpy(), flags=ops.workspace_status(ws))

    def optimize(self, prec, steps):
        m = self.model()
        kw = {} if self.base is None else dict(decoder_base=self.base, k_active=self.K)
        dec = self.packed if self.base is not None else self.dec
        _, trace = self.vlg.optimize_splines(m, dec, self.t, steps, M=self.M, draws=None if self.draws is None
                                             else self.draws[:steps], seed=self.seed, curve_id0=self.id0,
                                             precision=prec, return_trace=True, **kw)
        return m, trace


def per_curve_rel(x, ref):
    return float(np.abs(np.asarray(x, np.float64) / ref - 1).max())


def grad_err(out, ref):
    """Largest per-curve error of dE/domega, dE/da, dE/db, relative to the curve's largest reference entry."""
    N = ref["ga"].shape[0]
    scale = np.maximum.reduce([np.abs(ref[k]).reshape(N, -1).max(1) for k in ("gom", "ga", "gb")])
    errs = {k: float((np.abs(out[k] - ref[k]).reshape(N, -1).max(1) / scale).max()) for k in ("gom", "ga", "gb")}
    return errs


def energy_err(E, ref_E, prec):
    """Relative error per curve; the 11-bit modes: of sqrt(E), the geodesic length."""
    return per_curve_rel(np.sqrt(E / ref_E) if prec in ELEVEN_BIT else E / ref_E, 1.0)


def warn_context(name, prec):
    """More than 128 decoders on a tensor-core precision must warn (fallback to the fp32 kernel)."""
    if shape(name)[2] > TC_MAX_K and prec != "fp32":
        return pytest.warns(UserWarning, match="K <= 128")
    return warnings.catch_warnings()


def sweep_params():
    out = []
    for name, (N, T, K, M, *_rest) in CASES.items():
        for prec in PRECISIONS:
            if prec == "fp32" and M > FP32_MAX_M:
                continue                       # the fp32 kernel holds at most 4 samples (VLG_ERR_UNSUPPORTED)
            for mode in ("explicit", "counter"):
                out.append(pytest.param(name, prec, mode, id=f"{name}-{prec}-{mode}"))
    return out


# ------------------------------------------------------------------ GPU: regime sweep ----------------------------

@gpu
@pytest.mark.parametrize("name,prec,mode", sweep_params())
def test_launch_plan_against_fp64(vlg, name, prec, mode):
    """(a) the gradient launch, (b) the same numbers as the optimiser's first step, (c) the forward-only energy and
    length, (d) three optimiser steps -- against the sparse fp64 reference."""
    run = Run(vlg, name, mode)
    ref = case_reference(name, mode)
    tol = tolerances(name, prec)
    eff = effective_precision(name, prec)
    with warn_context(name, prec):
        g = run.grad(prec)
        f = run.forward(prec)
        m1, trace1 = run.optimize(prec, 1)
        mS, traceS = run.optimize(prec, STEPS)
    # (a)
    assert g["flags"] == 0 and f["flags"] == 0
    eE = energy_err(g["E"], ref["E"], eff)
    ge = grad_err(g, ref)
    # (c)
    eEf = energy_err(f["E"], ref["E"], eff)
    eL = per_curve_rel(f["L"], ref["L"])
    # (d)
    trace = traceS.cpu().numpy()
    eT = per_curve_rel(np.sqrt(trace / ref["trace"]) if eff in ELEVEN_BIT else trace / ref["trace"], 1.0)
    # Adam moves a coefficient by ~lr per step whatever its gradient's size, so a component whose fp64 gradient lies
    # below the fp32 gradient bound has no determined direction.  Of all cases here that is every component at T = 2
    # and nothing else: both points sit on the end points, where all basis functions vanish, and dE/domega is rounding
    # of the fp32 basis in the kernel and in the reference alike.  Such components only have to stay within Adam's
    # largest move.
    d_om = np.abs(mS.omega.cpu().numpy() - ref["omega_S"])
    scale = np.maximum.reduce([np.abs(ref[k]).reshape(run.N, -1).max(1) for k in ("gom", "ga", "gb")])
    resolved = np.abs(ref["gom"]) > TOL["fp32"]["G"] * scale[:, None, None]
    eO = float(d_om[resolved].max(initial=0.0))
    eO_free = float(d_om[~resolved].max(initial=0.0))
    print(f"\nERR {regime(name)} {name} {prec} {mode}: E {eE:.2e} Efwd {eEf:.2e} L {eL:.2e} "
          f"gom {ge['gom']:.2e} ga {ge['ga']:.2e} gb {ge['gb']:.2e} trace {eT:.2e} omega {eO:.2e} "
          f"(unresolved {int((~resolved).sum())}/{resolved.size}: {eO_free:.2e})")
    assert eE < tol["E"] and eEf < tol["E"] and eL < tol["L"]
    assert max(ge.values()) < tol["G"], ge
    # (b) the energy is the optimiser's first-step energy, bit for bit; dE/domega = adam_m / (1 - beta1) - penalty
    assert torch.equal(g["E_t"], trace1[0])
    c = run.c
    err_end = run.model()(run.t[-1:])[0].cpu().double().numpy() - c["b"].astype(np.float64)
    P1 = O.design_matrix(c["basis"].astype(np.float64), c["t"].astype(np.float64)[-1:], run.n_poly)[0]
    g_opt = m1.adam_m.double().cpu().numpy() / (1 - BETA1) - 2 * PENALTY * err_end[:, None, :] * P1[None, :, None]
    assert Hh.relerr(g["gom"], g_opt) < 1e-6
    # (d)
    assert eT < TRACE_TOL[eff] and eO < OMEGA_TOL[eff]
    assert eO_free < 2 * STEPS * LR + 1e-6


# ------------------------------------------------------------------ GPU: forced plans ----------------------------

@gpu
@pytest.mark.parametrize("prec", ["f16x3", "f16x3f", "f16", "tf32"])
@pytest.mark.parametrize("name", list(FORCED))
def test_every_home_and_grouping_gives_the_same_numbers(vlg, monkeypatch, name, prec):
    """The same inputs through every admissible plan (the host honours VLG_TC_XL2 / VLG_TC_G / VLG_TC_WINDOW on
    every call): each meets the fp64 bound; all groupings of the L2 home are bit-identical (DESIGN 4.2), gradients
    included; the shared-memory and L2 homes agree to 2e-6 where the arithmetic is fp32-grade."""
    run = Run(vlg, name, "counter")
    ref = case_reference(name, "counter")
    tol = tolerances(name, prec)
    res = {}
    for label, env in FORCED[name][1]:
        for k in ("VLG_TC_XL2", "VLG_TC_G", "VLG_TC_WINDOW"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        g, f = run.grad(prec), run.forward(prec)   # a plan the host rejects raises VlgError: the list is fixed
        assert g["flags"] == 0 and f["flags"] == 0, label
        eE, eEf, eL = energy_err(g["E"], ref["E"], prec), energy_err(f["E"], ref["E"], prec), per_curve_rel(f["L"], ref["L"])
        ge = grad_err(g, ref)
        print(f"\nPLAN {name} {label} {prec}: E {eE:.2e} Efwd {eEf:.2e} L {eL:.2e} gom {ge['gom']:.2e} "
              f"ga {ge['ga']:.2e} gb {ge['gb']:.2e}")
        assert eE < tol["E"] and eEf < tol["E"] and eL < tol["L"], label
        assert max(ge.values()) < tol["G"], (label, ge)
        res[label] = dict(g, Ef=f["E"], L=f["L"])
    keys = ("E", "gom", "ga", "gb", "Ef", "L")
    l2 = [lab for lab in res if lab.startswith("l2")]
    smem = [lab for lab in res if lab.startswith("smem")]
    if len(l2) > 1:
        for lab in l2[1:]:
            for k in keys:
                assert np.array_equal(res[lab][k], res[l2[0]][k]), (lab, k)
    if prec in ("f16x3", "f16x3f"):
        for s in smem:
            for lab in l2:
                a, b = res[s], res[lab]
                gap = dict(E=per_curve_rel(a["E"], b["E"]), Ef=per_curve_rel(a["Ef"], b["Ef"]),
                           L=per_curve_rel(a["L"], b["L"]))
                gap.update(grad_err(a, b))
                print(f"HOMES {name} {s} vs {lab} {prec}: " + " ".join(f"{k} {v:.2e}" for k, v in gap.items()))
                checked = ("E", "Ef", "L", "gom", "ga", "gb") if prec == "f16x3" else ("E", "Ef", "L")
                assert max(gap[k] for k in checked) < 2e-6, gap


# ------------------------------------------------------------------ GPU: output width ----------------------------

@gpu
@pytest.mark.parametrize("X", [1, 3, 49, 52])
@pytest.mark.parametrize("prec", ["fp32", "f16x3", "f16x3f"])
@pytest.mark.parametrize("name", ["r2_T2000_K10_M2", "r4_T256_K16_M3"])
def test_output_width(vlg, name, prec, X):
    """Decoders with X outputs (the kernels store 52-float rows and rely on zero padding past X): packing, the
    gradient launch, compute_energy_mc with the length and three optimiser steps against the fp64 reference."""
    run = Run(vlg, name, "explicit", X)
    assert run.packed.X == X
    ref = case_reference(name, "explicit", X)
    tol = TOL[prec]
    g = run.grad(prec)
    assert g["flags"] == 0
    E, L = vlg.compute_energy_mc(run.model(), run.dec, run.t, M=run.M, draws=run.draws[0], precision=prec,
                                 return_length=True)
    mS, trace = run.optimize(prec, STEPS)
    errs = dict(E=energy_err(g["E"], ref["E"], prec), Emc=energy_err(E.cpu().numpy(), ref["E"], prec),
                L=per_curve_rel(L.cpu().numpy(), ref["L"]), trace=per_curve_rel(trace.cpu().numpy(), ref["trace"]),
                omega=float(np.abs(mS.omega.cpu().numpy() - ref["omega_S"]).max()))
    errs.update(grad_err(g, ref))
    print(f"\nWIDTH {name} X={X} {prec}: " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    assert errs["E"] < tol["E"] and errs["Emc"] < tol["E"] and errs["L"] < tol["L"]
    assert max(errs[k] for k in ("gom", "ga", "gb")) < tol["G"]
    assert errs["trace"] < TRACE_TOL[prec] and errs["omega"] < OMEGA_TOL[prec]


@gpu
@pytest.mark.parametrize("X", [1, 3, 49, 52])
def test_ensemble_std_norm_output_width(vlg, X):
    W = decoder_arrays(10, X)
    dec = vlg.DecoderEnsemble.from_arrays(*[W[k] for k in Hh.DEC_KEYS], "cuda")
    grid = np.random.default_rng(X).uniform(-3, 3, (777, 2)).astype(np.float32)
    s = vlg.ensemble_std_norm(dec, torch.tensor(grid, device="cuda")).cpu().numpy()
    ref = O.ensemble_std_norm(grid.astype(np.float64), Hh.decoder_list(W, 10, np.float64))
    err = float((np.abs(s - ref) / np.maximum(ref, 1e-3 * ref.max())).max())
    print(f"\nSTD X={X}: {err:.2e}")
    assert err < 2e-5


# ------------------------------------------------------------------ GPU: spline-point backward --------------------

@gpu
@pytest.mark.parametrize("N,T,n_poly,grid", [(1, 100, 4, "uniform"), (3, 1, 4, "uniform"), (2, 100003, 4, "uniform"),
                                             (3, 257, 1, "uniform"), (3, 257, 8, "uniform"), (3, 300, 8, "knots")])
def test_spline_points_backward_edges(vlg, N, T, n_poly, grid):
    """vlg_spline_points_backward (the autograd path of GeodesicSplineBatch.forward) against fp64 autograd: one curve,
    one point, many reduction chunks, a single segment, the largest n_poly, a non-uniform grid."""
    from vlg_b200 import api
    rng = np.random.default_rng(T + N)
    t = nonuniform_grid(T, n_poly) if grid == "knots" else Hh.tgrid(T)
    basis = api.construct_nullspace_basis(n_poly)[0]
    a, b = rng.uniform(-2, 2, (N, 2)).astype(np.float32), rng.uniform(-2, 2, (N, 2)).astype(np.float32)
    om = (0.1 * rng.normal(size=(N, n_poly + 1, 2))).astype(np.float32)
    w = (rng.normal(size=(T, N, 2)) + 0.5).astype(np.float32)
    model = vlg.GeodesicSplineBatch(torch.tensor(a, device="cuda"), torch.tensor(b, device="cuda"), basis.cuda(),
                                    torch.tensor(om, device="cuda"), n_poly)
    for x in (model.omega, model.a, model.b):
        x.requires_grad_(True)
    (model(torch.tensor(t, device="cuda")) * torch.tensor(w, device="cuda")).sum().backward()
    ta = torch.tensor(a, dtype=F64, requires_grad=True)
    tb = torch.tensor(b, dtype=F64, requires_grad=True)
    sb = TP.SplineBatch(ta, tb, basis.double(), torch.tensor(om, dtype=F64), n_poly)
    (sb(torch.tensor(t, dtype=F64)) * torch.tensor(w, dtype=F64)).sum().backward()
    for name, x, ref in (("omega", model.omega, sb.omega), ("a", model.a, ta), ("b", model.b, tb)):
        err = Hh.relerr(x.grad.cpu().numpy(), ref.grad.numpy())
        print(f"\nSPLINE-BWD N={N} T={T} n_poly={n_poly} {grid} d{name}: {err:.2e}")
        assert err < 1e-6, name
