"""GPU (B200): the CUDA path, called through the C ABI (ctypes via vlg_b200.ops), against the
CPU oracle and the committed reference goldens on identical inputs and decoder draws.

Tolerances (north_star): fp32 variant <= 1e-4 relative per-step energy; the tests assert a much
tighter bound where the arithmetic allows it and say so."""
import numpy as np
import pytest
import torch

from oracle import geodesic_oracle as O
from tests import helpers as Hh

pytestmark = pytest.mark.gpu

FP32_STEP_TOL = 1e-4  # north_star: relative per-step energy, fp32 variant


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
    ens = vlg.DecoderEnsemble.from_arrays(*[arrs[k] for k in Hh.DEC_KEYS], dev)
    return ens[:K]


MC_CASES = ["ens_seed12_euclid", "ens_seed12_entropy", "ens_seed12_cov_k3", "synth_np8_T256", "synth_np4_T130"]


@pytest.mark.parametrize("tag", MC_CASES)
def test_fp32_steps_match_reference_goldens(vlg, tag):
    """Explicit recorded draws, S Adam steps: per-step energy, then omega / m / v."""
    g = Hh.load(tag)
    K, T, M, S = int(g["K"]), int(g["T"]), int(g["M"]), int(g["steps"])
    draws = Hh.regen_draws(g)[:S]
    model = make_model(vlg, g)
    dec = make_decoders(vlg, g, K)
    t = torch.linspace(0, 1, T, device="cuda")
    e_last, trace = vlg.optimize_splines(model, dec, t, S, M=M, draws=draws, precision="fp32", return_trace=True)
    trace = trace.cpu().numpy()
    rel = np.abs(trace / g["energy_f64"] - 1).max()
    assert rel < FP32_STEP_TOL
    assert rel < 5e-6, f"fp32 kernel should track the fp64 reference far inside the stated tolerance, got {rel}"
    assert np.abs(trace / g["energy_f32"] - 1).max() < 5e-6
    assert np.array_equal(e_last.cpu().numpy(), trace[-1])
    assert np.abs(model.omega.cpu().numpy() - g["omega_f64"]).max() < 5e-6
    assert Hh.relerr(model.adam_m.cpu().numpy(), g["m_f64"]) < 2e-5
    assert Hh.relerr(model.adam_v.cpu().numpy(), g["v_f64"]) < 4e-5
    assert model.step_count == S


@pytest.mark.parametrize("tag", MC_CASES)
def test_3term_tensor_core_mode_meets_the_fp32_tolerance(vlg, tag):
    """f16x3 (hi/lo fp16 operands, three MMAs per product, fp32 accumulate): the tensor-core mode that meets the
    fp32 variant's bound -- <= 1e-4 relative per-step energy -- with a wide margin."""
    g = Hh.load(tag)
    K, T, M, S = int(g["K"]), int(g["T"]), int(g["M"]), int(g["steps"])
    if M > 2:
        pytest.skip("tensor-core path is built for M <= 2 (shared-memory budget)")
    draws = Hh.regen_draws(g)[:S]
    model = make_model(vlg, g)
    dec = make_decoders(vlg, g, K)
    t = torch.linspace(0, 1, T, device="cuda")
    _, trace = vlg.optimize_splines(model, dec, t, S, M=M, draws=draws, precision="f16x3", return_trace=True)
    rel = np.abs(trace.cpu().numpy() / g["energy_f64"] - 1).max()
    print(f"{tag}: f16x3 max rel per-step energy err {rel:.2e}")
    assert rel < FP32_STEP_TOL
    assert rel < 1e-5, rel
    assert np.abs(model.omega.cpu().numpy() - g["omega_f64"]).max() < 2e-5
    assert Hh.relerr(model.adam_m.cpu().numpy(), g["m_f64"]) < 2e-4


def test_fp32_gradient_via_first_adam_moment(vlg):
    """After one step from zero state m = (1-beta1) * grad: checks d(loss)/d(omega)."""
    g = Hh.load("ens_seed12_euclid")
    draws = Hh.regen_draws(g)[:1]
    model = make_model(vlg, g)
    dec = make_decoders(vlg, g, 10)
    t = torch.linspace(0, 1, 2000, device="cuda")
    vlg.optimize_splines(model, dec, t, 1, M=2, draws=draws, precision="fp32")
    grad = model.adam_m.cpu().numpy().astype(np.float64) / (1 - 0.9)
    assert Hh.relerr(grad, g["grad0_f64"]) < 2e-5
    assert np.abs(model.omega.cpu().numpy() - g["omega1_f64"]).max() < 1e-6


def test_forward_energy_and_spline_points(vlg):
    g = Hh.load("ens_seed12_entropy")
    draws = Hh.regen_draws(g)[:1]
    model = make_model(vlg, g)
    dec = make_decoders(vlg, g, 10)
    t = torch.linspace(0, 1, 2000, device="cuda")
    E = vlg.compute_energy_mc(model, dec, t, M=2, draws=draws, precision="fp32").cpu().numpy()
    assert np.abs(E / g["energy_f64"][0] - 1).max() < 5e-6
    z = model(t).cpu().numpy()
    zo = O.spline_points(g["a"], g["b"], g["omega_init"], g["basis"], Hh.tgrid(2000), int(g["n_poly"]))
    assert np.abs(z - zo).max() < 2e-6


def test_counter_draws_match_oracle_stream(vlg):
    """draws=NULL: the in-kernel Philox stream equals oracle.counter_draws (same energies)."""
    g = Hh.load("synth_np8_T256")
    K, T, M = int(g["K"]), int(g["T"]), int(g["M"])
    N = g["a"].shape[0]
    model = make_model(vlg, g)
    dec = make_decoders(vlg, g, K)
    t = torch.linspace(0, 1, T, device="cuda")
    seed, id0, S = 0x1234567811, 1000, 3
    _, trace = vlg.optimize_splines(model, dec, t, S, M=M, seed=seed, curve_id0=id0, precision="fp32", return_trace=True)
    draws = np.stack([O.counter_draws(seed, np.arange(N) + id0, s, T, M, K) for s in range(S)])
    decs = Hh.decoder_list(Hh.decoder_arrays(g), K, np.float64)
    r = O.optimize_steps(g["a"].astype(np.float64), g["b"].astype(np.float64), g["omega_init"].astype(np.float64),
                         g["basis"].astype(np.float64), Hh.tgrid(T, np.float64), int(g["n_poly"]), decs, draws, S)
    assert np.abs(trace.cpu().numpy() / r["energy"] - 1).max() < 5e-6
    assert np.abs(model.omega.cpu().numpy() - r["omega"]).max() < 5e-6


def test_results_do_not_depend_on_sharding_or_chunking(vlg):
    """Curves are independent and draws are keyed on the global curve id: splitting the pair
    list (multi-GPU sharding) or the step range (chunked launches) is bit-identical."""
    g = Hh.load("synth_np4_T130")
    K, T, M = int(g["K"]), int(g["T"]), int(g["M"])
    N = g["a"].shape[0]
    dec = make_decoders(vlg, g, K)
    t = torch.linspace(0, 1, T, device="cuda")
    full = make_model(vlg, g)
    e_full = vlg.optimize_splines(full, dec, t, 4, M=M, seed=9, curve_id0=50, precision="fp32")
    # two shards
    parts = []
    for lo, hi in ((0, 2), (2, N)):
        sub = {k: (v[lo:hi] if k in ("a", "b", "omega_init") else v) for k, v in g.items()}
        m = make_model(vlg, sub)
        e = vlg.optimize_splines(m, dec, t, 4, M=M, seed=9, curve_id0=50 + lo, precision="fp32")
        parts.append((m.omega, e))
    assert torch.equal(torch.cat([p[0] for p in parts]), full.omega)
    assert torch.equal(torch.cat([p[1] for p in parts]), e_full)
    # two step chunks
    ch = make_model(vlg, g)
    vlg.optimize_splines(ch, dec, t, 3, M=M, seed=9, curve_id0=50, precision="fp32")
    e2 = vlg.optimize_splines(ch, dec, t, 1, M=M, seed=9, curve_id0=50, precision="fp32")
    assert torch.equal(ch.omega, full.omega) and torch.equal(e2, e_full)


@pytest.mark.parametrize("prec", ["fp32", "f16x3", "f16x3f"])
def test_single_decoder_path(vlg, prec):
    """BASELINE config 2: deterministic energy, 6 steps, then the poly-line length.  The 3-term tensor-core mode holds
    the same bound as the fp32 kernel here (the single-term modes cannot: 11-bit operands, SURVEY hard part 1)."""
    g = Hh.load("single_seed123")
    model = make_model(vlg, g)
    dec = make_decoders(vlg, g, 1)
    t = torch.linspace(0, 1, 2000, device="cuda")
    E0 = vlg.compute_energy(model, dec, t, precision=prec).cpu().numpy()
    # sums of tiny differences of large numbers: fp32 noise of the reference itself is ~1e-4 here
    e0 = np.abs(E0 / g["energy_f64"][0] - 1).max()
    assert e0 < 5e-4
    S = int(g["steps"])
    _, trace = vlg.optimize_splines(model, dec, t, S, M=1, precision=prec, return_trace=True)
    et = np.abs(trace.cpu().numpy() / g["energy_f64"] - 1).max()
    assert et < 5e-4
    L = vlg.compute_geodesic_lengths(model, dec, t, precision=prec).cpu().numpy()
    el = np.abs(L / g["length_f64"] - 1).max()
    print(f"\nsingle decoder [{prec}]: energy {e0:.1e}, {S}-step energies {et:.1e}, poly-line length {el:.1e} (rel. to fp64)")
    assert el < 2e-4


def test_std_field(vlg):
    g = Hh.load("std_field_seed12")
    dec = make_decoders(vlg, Hh.load("evae_seed12_decoders"), 10)
    s = vlg.ensemble_std_norm(dec, torch.tensor(g["grid"], device="cuda")).cpu().numpy()
    assert np.abs(s / g["std_norm_f64"] - 1).max() < 2e-5
    s3 = vlg.ensemble_std_norm(dec[:3], torch.tensor(g["grid"][:77], device="cuda")).cpu().numpy()
    ref3 = O.ensemble_std_norm(g["grid"][:77].astype(np.float64),
                               Hh.decoder_list(Hh.load("evae_seed12_decoders"), 3, np.float64))
    assert np.abs(s3 / ref3 - 1).max() < 2e-5


def test_spline_fit(vlg):
    g = Hh.load("lbfgs_fit")
    paths = [torch.tensor(g["targets"][i, :L]) for i, L in enumerate(g["lens"])]
    a, b, om = vlg.fit_splines_to_paths(paths, torch.tensor(g["basis"]), 4, "cuda")
    for i, L in enumerate(g["lens"]):
        ref = O.fit_spline_to_path(g["targets"][i, :L], g["basis"], 4)
        assert np.abs(om[i].cpu().numpy() - ref).max() < 2e-5
        assert np.abs(om[i].cpu().numpy() - g["omega_lbfgs"][i]).max() < 5e-3
        assert np.array_equal(a[i].cpu().numpy(), g["targets"][i, 0])
        assert np.array_equal(b[i].cpu().numpy(), g["targets"][i, L - 1])


@pytest.mark.parametrize("T,N,K,M,n_poly", [(2, 1, 1, 1, 1), (3, 2, 2, 2, 2), (128, 3, 3, 4, 4), (129, 2, 5, 1, 8),
                                           (255, 1, 16, 2, 4)])
def test_edge_shapes_against_oracle(vlg, T, N, K, M, n_poly):
    """Ragged / minimal sizes: T=2 (one segment), tile boundaries (128, 129, 255), M up to 4,
    K up to 16, single curve."""
    rng = np.random.default_rng(T * 31 + K)
    torch.manual_seed(T)
    W = dict(W1=rng.normal(size=(K, 128, 2)) * 0.7, b1=rng.normal(size=(K, 128)) * 0.3,
             W2=rng.normal(size=(K, 128, 128)) * 0.09, b2=rng.normal(size=(K, 128)) * 0.1,
             W3=rng.normal(size=(K, 50, 128)) * 0.09, b3=rng.normal(size=(K, 50)) * 0.1)
    W = {k: v.astype(np.float32) for k, v in W.items()}
    basis, _ = vlg.construct_nullspace_basis(n_poly)
    g = dict(a=rng.uniform(-3, 3, (N, 2)).astype(np.float32), b=rng.uniform(-3, 3, (N, 2)).astype(np.float32),
             omega_init=(0.1 * rng.normal(size=(N, n_poly + 1, 2))).astype(np.float32), basis=basis.numpy(),
             n_poly=n_poly, **W)
    S = 2
    draws = rng.integers(0, K, size=(S, M, 2, T - 1, N))
    model = make_model(vlg, g)
    dec = make_decoders(vlg, g, K)
    t = torch.linspace(0, 1, T, device="cuda")
    _, trace = vlg.optimize_splines(model, dec, t, S, M=M, draws=draws, precision="fp32", return_trace=True)
    r = O.optimize_steps(g["a"].astype(np.float64), g["b"].astype(np.float64), g["omega_init"].astype(np.float64),
                         g["basis"].astype(np.float64), Hh.tgrid(T, np.float64), n_poly,
                         Hh.decoder_list(W, K, np.float64), draws, S)
    assert np.abs(trace.cpu().numpy() / r["energy"] - 1).max() < 1e-5
    assert np.abs(model.omega.cpu().numpy() - r["omega"]).max() < 5e-6


def test_full_size_config1_teacher_forced(vlg):
    """BASELINE config 1 at full size (45 curves, T=2000, K=10, M=2): one step, oracle fp64."""
    s = Hh.load("splines_seed12_euclidean_10")
    g = dict(a=s["a"], b=s["b"], omega_init=s["omega_init"], basis=s["basis"], n_poly=int(s["n_poly"]))
    N, T, K, M = 45, 2000, 10, 2
    gen = torch.Generator().manual_seed(2024)
    draws = torch.randint(0, K, (1, M, 2, T - 1, N), generator=gen).numpy()
    model = make_model(vlg, g)
    dec = make_decoders(vlg, Hh.load("evae_seed12_decoders"), K)
    t = torch.linspace(0, 1, T, device="cuda")
    E = vlg.optimize_splines(model, dec, t, 1, M=M, draws=draws, precision="fp32").cpu().numpy()
    decs = Hh.decoder_list(Hh.load("evae_seed12_decoders"), K, np.float64)
    r = O.optimize_steps(g["a"].astype(np.float64), g["b"].astype(np.float64), g["omega_init"].astype(np.float64),
                         g["basis"].astype(np.float64), Hh.tgrid(T, np.float64), 4, decs, draws, 1)
    assert np.abs(E / r["energy"][0] - 1).max() < 5e-6
    assert np.abs(model.omega.cpu().numpy() - r["omega"]).max() < 2e-6
    # sanity against the reference's committed result: same order of magnitude of sqrt(E)
    assert 0.3 < np.median(np.sqrt(E) / s["committed_geodesic_length"]) < 3.0


def test_errors_are_loud(vlg):
    g = Hh.load("synth_np4_T130")
    model = make_model(vlg, g)
    dec = make_decoders(vlg, g, 4)
    t = torch.linspace(0, 1, 130, device="cuda")
    with pytest.raises(vlg.VlgError):
        vlg.optimize_splines(model, dec, t, 1, M=9, precision="fp32")        # M too large for the fp32 kernel
    with pytest.warns(UserWarning):                                          # one decoder: tf32 request served by the fp32 kernel
        e3 = vlg.optimize_splines(make_model(vlg, g), dec[:1], t, 1, M=3, seed=1, precision="tf32")
    assert torch.equal(e3, vlg.optimize_splines(make_model(vlg, g), dec[:1], t, 1, M=3, seed=1, precision="fp32"))
    with pytest.raises(vlg.VlgError):
        vlg.optimize_splines(model, dec, t.cpu(), 1, M=1, precision="fp32")  # CPU tensor
    with pytest.raises(vlg.VlgError):
        vlg.optimize_splines(model, dec, t, 1, M=1, draws=np.zeros((1, 1, 2, 5, 5)), precision="fp32")
    N = g["a"].shape[0]
    with pytest.raises(vlg.VlgError):                                        # draw index 4 with 4 active decoders
        vlg.optimize_splines(make_model(vlg, g), dec, t, 1, M=1, draws=np.full((1, 1, 2, 129, N), 4), precision="fp32")
    with pytest.raises(vlg.VlgError):
        vlg.optimize_splines(make_model(vlg, g), dec, t, 1, M=1, precision="bf16")


@pytest.mark.parametrize("prec", ["fp32", "f16", "f16x3", "tf32"])
def test_kernel_status_word_reports_bad_draws_and_overflow(vlg, prec):
    """The C ABI itself (no host-side validation): an out-of-range explicit draw is clamped and flagged, and
    a non-finite result (fp16 operand overflow, or an omega the Adam step made non-finite) is flagged --
    vlg_workspace_status returns VLG_ERR_NUMERIC."""
    from vlg_b200 import ops, api
    g = Hh.load("synth_np4_T130")
    N, T, K, M = g["a"].shape[0], 130, 4, 2
    dec = make_decoders(vlg, g, K)
    code = ops.PRECISIONS[prec]
    t = torch.linspace(0, 1, T, device="cuda")

    def launch(dec_, draws, lr=1e-3):
        m = make_model(vlg, g)
        ws = api._workspace(m, dec_, T, M, code)
        e = torch.empty(N, device="cuda")
        ops.optimize_steps(dec_.packed, dec_.K, dec_.X, len(dec_), 4, M, 1, 0, m.a, m.b, m.omega, m.adam_m, m.adam_v,
                           m.basis, t, draws, None, 0, 0, lr, 0.9, 0.999, 1e-8, 1000.0, e, None, code, ws)
        return ops.workspace_status(ws), e

    assert launch(dec, None)[0] == 0
    bad = torch.full((N, 1, M, 2, T - 1), 200, dtype=torch.uint8, device="cuda")
    flags, e = launch(dec, bad)
    assert flags & ops.STATUS_BAD_DRAW and bool(torch.isfinite(e).all())     # clamped to decoder K-1, memory-safe
    flags, e = launch(dec, None, lr=float("inf"))     # the energy before the step is finite, the stepped omega is not
    assert flags & ops.STATUS_NONFINITE and bool(torch.isfinite(e).all())
    # decoders whose hidden activations exceed the fp16 range
    arrs = {k: v.copy() for k, v in Hh.decoder_arrays(g).items()}
    arrs["W2"] = arrs["W2"] * 3.0e4
    big = vlg.DecoderEnsemble.from_arrays(*[arrs[k] for k in Hh.DEC_KEYS], "cuda")[:K]
    flags, e = launch(big, None)
    if prec in ("f16", "f16x3"):
        assert flags & ops.STATUS_NONFINITE
        with pytest.raises(vlg.VlgError, match="fp16 range"):
            vlg.optimize_splines(make_model(vlg, g), big, t, 1, M=M, precision=prec)
    else:
        assert flags == 0 and bool(torch.isfinite(e).all())


@pytest.mark.parametrize("tc", ["tf32", "f16", "f16x3"])
def test_split_row_lists_are_deterministic(vlg, tc):
    """Few decoders and long windows: every decoder is drawn by far more than 128 points of a window, so
    each row list is split into several 128-row items that run on DIFFERENT chains.  Item membership is
    by point order (not by thread arrival order), so repeated runs, a different launch shape and any
    sharding give bit-identical results (the round-1 kernel failed exactly this)."""
    rng = np.random.default_rng(7)
    K, T, N, S = 2, 600, 300, 3
    W = dict(W1=rng.normal(size=(K, 128, 2)) * 0.7, b1=rng.normal(size=(K, 128)) * 0.3,
             W2=rng.normal(size=(K, 128, 128)) * 0.09, b2=rng.normal(size=(K, 128)) * 0.1,
             W3=rng.normal(size=(K, 50, 128)) * 0.09, b3=rng.normal(size=(K, 50)) * 0.1)
    dec = make_decoders(vlg, {k: v.astype(np.float32) for k, v in W.items()}, K)
    basis, _ = vlg.construct_nullspace_basis(4)
    a = torch.tensor(rng.uniform(-3, 3, (N, 2)), dtype=torch.float32)
    b = torch.tensor(rng.uniform(-3, 3, (N, 2)), dtype=torch.float32)
    om = torch.tensor(0.1 * rng.normal(size=(N, 5, 2)), dtype=torch.float32)
    t = torch.linspace(0, 1, T, device="cuda")

    def run(lo, hi):
        m = vlg.GeodesicSplineBatch(a[lo:hi].cuda(), b[lo:hi].cuda(), basis.cuda(), om[lo:hi].cuda(), 4)
        e = vlg.optimize_splines(m, dec, t, S, M=2, seed=9, curve_id0=lo, precision=tc)
        return m.omega.clone(), e.clone()

    ref_om, ref_e = run(0, N)
    assert bool(torch.isfinite(ref_e).all())
    for _ in range(4):                                   # run to run
        o, e = run(0, N)
        assert torch.equal(o, ref_om) and torch.equal(e, ref_e)
    for parts in (2, 7):                                 # shard to shard
        from vlg_b200.sharding import shard_range
        oms, es = zip(*[run(*shard_range(N, r, parts)) for r in range(parts)])
        assert torch.equal(torch.cat(oms), ref_om) and torch.equal(torch.cat(es), ref_e)


# ---------------------------------------------------------------------------------------------
# tensor-core variants (tcgen05 kind::tf32, and kind::f16 with fp16 operands -- the same 11-bit
# significand).  north_star tolerance: <= 1e-3 relative on geodesic lengths (sqrt(E)), i.e. <= 2e-3
# on energies.
# ---------------------------------------------------------------------------------------------
TF32_LENGTH_TOL = 1e-3
TC_PRECISIONS = ["tf32", "f16", "f16x3", "f16x3f"]


@pytest.mark.parametrize("tag", ["ens_seed12_euclid", "ens_seed12_entropy", "ens_seed12_cov_k3", "synth_np8_T256",
                                 "synth_np4_T130"])
@pytest.mark.parametrize("tc", TC_PRECISIONS)
def test_tf32_steps_track_reference(vlg, tag, tc):
    g = Hh.load(tag)
    K, T, M, S = int(g["K"]), int(g["T"]), int(g["M"]), int(g["steps"])
    if M > 2:
        pytest.skip("tensor-core path is built for M <= 2 (shared-memory budget)")
    draws = Hh.regen_draws(g)[:S]
    model = make_model(vlg, g)
    dec = make_decoders(vlg, g, K)
    t = torch.linspace(0, 1, T, device="cuda")
    e_last, trace = vlg.optimize_splines(model, dec, t, S, M=M, draws=draws, precision=tc, return_trace=True)
    trace = trace.cpu().numpy()
    len_rel = np.abs(np.sqrt(trace / g["energy_f64"]) - 1).max()
    assert len_rel < TF32_LENGTH_TOL, len_rel
    # gradient quality: first Adam moment after S steps stays close to the fp64 one
    assert Hh.relerr(model.adam_m.cpu().numpy(), g["m_f64"]) < 3e-2
    # Adam normalises the gradient, so near-zero gradient components turn tiny errors into
    # +-lr-sized steps: after S steps omega may differ by a fraction of S*lr = S*1e-3
    assert np.abs(model.omega.cpu().numpy() - g["omega_f64"]).max() < 0.25 * S * 1e-3
    print(f"{tag}: {tc} max rel length err {len_rel:.2e}")


@pytest.mark.parametrize("tc", TC_PRECISIONS)
def test_tf32_forward_energy_full_size(vlg, tc):
    s = Hh.load("splines_seed12_entropy_10")
    g = dict(a=s["a"], b=s["b"], omega_init=s["omega_init"], basis=s["basis"], n_poly=int(s["n_poly"]))
    N, T, K, M = 45, 2000, 10, 2
    model = make_model(vlg, g)
    dec = make_decoders(vlg, Hh.load("evae_seed12_decoders"), K)
    t = torch.linspace(0, 1, T, device="cuda")
    e32 = vlg.compute_energy_mc(model, dec, t, M=M, seed=3, step=7, precision="fp32").cpu().numpy()
    etc = vlg.compute_energy_mc(model, dec, t, M=M, seed=3, step=7, precision=tc).cpu().numpy()
    assert np.abs(np.sqrt(etc / e32) - 1).max() < TF32_LENGTH_TOL


@pytest.mark.parametrize("prec,tol", [("fp32", 2e-5), ("tf32", TF32_LENGTH_TOL), ("f16", TF32_LENGTH_TOL), ("f16x3", 2e-5), ("f16x3f", 1e-4)])
def test_final_length_after_150_steps(vlg, prec, tol):
    """Long horizon (free-running, not teacher-forced): final sqrt(E) against the reference's own
    fp64 run with the same recorded draws.  The reference's fp32-vs-fp64 gap is printed beside it."""
    g = Hh.load("ens_seed12_long")
    S = int(g["long_steps"])
    draws = Hh.regen_draws(g)[:S]
    model = make_model(vlg, g)
    dec = make_decoders(vlg, Hh.load("evae_seed12_decoders"), 10)
    t = torch.linspace(0, 1, 2000, device="cuda")
    _, trace = vlg.optimize_splines(model, dec, t, S, M=2, draws=draws, precision=prec, return_trace=True)
    trace = trace.cpu().numpy()
    ref = g["long_energy_f64"]
    gap_ref32 = np.abs(np.sqrt(g["long_energy_f32"][-1] / ref[-1]) - 1).max()
    ours = np.abs(np.sqrt(trace[-1] / ref[-1]) - 1).max()
    print(f"final-length rel err after {S} steps: {prec} kernel {ours:.2e}; reference fp32 vs fp64 {gap_ref32:.2e}")
    assert ours < tol
    assert np.abs(np.sqrt(trace / ref) - 1).max() < tol * 2


@pytest.mark.parametrize("T,N,K,M,n_poly", [(2, 1, 1, 1, 1), (3, 2, 2, 2, 2), (128, 3, 3, 2, 4), (255, 2, 5, 1, 8),
                                           (256, 1, 16, 2, 4), (257, 2, 4, 2, 4), (600, 3, 1, 1, 4), (513, 150, 7, 2, 4),
                                           (300, 3, 6, 3, 4), (700, 2, 10, 4, 4), (130, 2, 3, 4, 2), (256, 9, 100, 2, 8)])
@pytest.mark.parametrize("tc", TC_PRECISIONS)
def test_tf32_edge_shapes_against_fp32_kernel(vlg, T, N, K, M, n_poly, tc):
    """Window boundaries (255/256/257 points), a decoder drawn by more than 128 points of a window
    (K=1: two 128-row items per window), a single segment, more curves than SMs (persistent CTAs
    walk several curves), K up to 100, more than two MC samples (the tensor-core kernel works through them in blocks
    of two; the reference exposes --mc-samples freely, src/optimize.py:232).  Compared against the fp32 kernel on
    identical draws."""
    rng = np.random.default_rng(T * 131 + K)
    W = dict(W1=rng.normal(size=(K, 128, 2)) * 0.7, b1=rng.normal(size=(K, 128)) * 0.3,
             W2=rng.normal(size=(K, 128, 128)) * 0.09, b2=rng.normal(size=(K, 128)) * 0.1,
             W3=rng.normal(size=(K, 50, 128)) * 0.09, b3=rng.normal(size=(K, 50)) * 0.1)
    W = {k: v.astype(np.float32) for k, v in W.items()}
    basis, _ = vlg.construct_nullspace_basis(n_poly)
    g = dict(a=rng.uniform(-3, 3, (N, 2)).astype(np.float32), b=rng.uniform(-3, 3, (N, 2)).astype(np.float32),
             omega_init=(0.1 * rng.normal(size=(N, n_poly + 1, 2))).astype(np.float32), basis=basis.numpy(),
             n_poly=n_poly, **W)
    S = 2
    dec = make_decoders(vlg, g, K)
    t = torch.linspace(0, 1, T, device="cuda")
    res = {}
    for prec in ("fp32", tc):
        model = make_model(vlg, g)
        _, trace = vlg.optimize_splines(model, dec, t, S, M=M, seed=11, curve_id0=5, precision=prec, return_trace=True)
        e, ln = vlg.compute_energy_mc(model, dec, t, M=M, seed=11, step=S, curve_id0=5, precision=prec,
                                      return_length=True)
        res[prec] = (trace.cpu().numpy(), model.omega.cpu().numpy(), e.cpu().numpy(), ln.cpu().numpy())
    # with random weights and few decoders the energies are single-decoder-like (differences of nearby
    # outputs), where TF32 is at its worst: allow 2e-2 on energies here; the real-checkpoint cases above
    # carry the 1e-3 length bound
    # K = 1 is the single-decoder energy (sum of tiny differences of large outputs): TF32 is known to be
    # inadequate there (SURVEY hard part 1: ~13 % mean error) -- that path is served by the fp32 kernel;
    # here it only has to be structurally right (same order of magnitude)
    tol = 0.5 if K == 1 else 2e-2
    assert np.abs(res[tc][0] / res["fp32"][0] - 1).max() < tol
    assert np.abs(res[tc][2] / res["fp32"][2] - 1).max() < tol
    assert np.abs(res[tc][3] / res["fp32"][3] - 1).max() < tol
    # Adam's first steps move every coefficient by ~lr whatever the gradient size, so a sign flip of a
    # near-zero gradient component costs up to 2*lr per step; frequent for K = 1 (noisy TF32 gradient)
    assert np.abs(res[tc][1] - res["fp32"][1]).max() < (2.0 if K == 1 else 0.25) * S * 1e-3 + 1e-6


@pytest.mark.parametrize("M", [3, 4])
def test_more_than_two_mc_samples_fp32_grade(vlg, M):
    """M > 2 on the tensor-core kernel (blocks of two samples), 3-term mode: fp32-grade agreement with the fp32
    kernel on the real ensemble, energies AND the omega after a few Adam steps; same draw stream (Philox keyed on the
    sample pair)."""
    g = Hh.load("ens_seed12_euclid")
    K, T = int(g["K"]), 500
    dec = make_decoders(vlg, g, K)
    t = torch.linspace(0, 1, T, device="cuda")
    res = {}
    for prec in ("fp32", "f16x3"):
        model = make_model(vlg, g)
        _, trace = vlg.optimize_splines(model, dec, t, 4, M=M, seed=3, precision=prec, return_trace=True)
        res[prec] = (trace.cpu().numpy(), model.omega.cpu().numpy())
    rel = np.abs(res["f16x3"][0] / res["fp32"][0] - 1).max()
    print(f"\nM={M}: f16x3 vs fp32 kernel, per-step energy max rel {rel:.2e}")
    assert rel < 2e-5
    assert np.abs(res["f16x3"][1] - res["fp32"][1]).max() < 2e-4


def test_six_mc_samples_against_the_oracle(vlg):
    """M = 6 (three sample blocks; beyond what the fp32 kernel holds) with explicit draws, 3-term mode, against the
    fp64 oracle: per-step energies of 3 Adam steps."""
    from oracle import geodesic_oracle as O
    g = Hh.load("synth_np4_T130")
    K, T, M, S = int(g["K"]), int(g["T"]), 6, 3
    N = g["a"].shape[0]
    draws = np.random.default_rng(5).integers(0, K, size=(S, M, 2, T - 1, N))
    arrs = Hh.decoder_arrays(g)
    ref = O.optimize_steps(g["a"].astype(np.float64), g["b"].astype(np.float64), g["omega_init"].astype(np.float64),
                           g["basis"].astype(np.float64), Hh.tgrid(T, np.float64), int(g["n_poly"]),
                           Hh.decoder_list(arrs, K, np.float64), draws, S)
    model = make_model(vlg, g)
    _, trace = vlg.optimize_splines(model, make_decoders(vlg, g, K), torch.linspace(0, 1, T, device="cuda"), S, M=M,
                                    draws=draws, precision="f16x3", return_trace=True)
    rel = np.abs(trace.cpu().numpy() / ref["energy"] - 1).max()
    print(f"\nM=6, f16x3 vs fp64 oracle: per-step energy max rel {rel:.2e}")
    assert rel < 2e-5
    assert np.abs(model.omega.cpu().numpy() - ref["omega"]).max() < 2e-5


@pytest.mark.parametrize("tc", TC_PRECISIONS)
def test_tf32_is_deterministic_and_shard_independent(vlg, tc):
    g = Hh.load("ens_seed12_entropy")
    dec = make_decoders(vlg, g, 10)
    t = torch.linspace(0, 1, 2000, device="cuda")
    outs = []
    for _ in range(2):
        m = make_model(vlg, g)
        e = vlg.optimize_splines(m, dec, t, 2, M=2, seed=5, curve_id0=40, precision=tc)
        outs.append((m.omega.clone(), e.clone()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    sub = {k: (v[2:5] if k in ("a", "b", "omega_init") else v) for k, v in g.items()}
    m = make_model(vlg, sub)
    e = vlg.optimize_splines(m, dec, t, 2, M=2, seed=5, curve_id0=42, precision=tc)
    assert torch.equal(m.omega, outs[0][0][2:5]) and torch.equal(e, outs[0][1][2:5])


def test_config5_shape_k64_npoly8_t256(vlg):
    """BASELINE config 5 shapes at a size the oracle finishes instantly: 64-decoder ensemble with default
    nn.Linear init, n_poly 8, T = 256 (the fp32 kernel keeps its ReLU masks in the workspace for K this
    large; the tensor-core kernel runs one 256-point window per curve)."""
    import torch.nn as nn
    torch.manual_seed(0)
    K, N, T, n_poly, M, S = 64, 20, 256, 8, 2, 2
    nets = [nn.Sequential(nn.Linear(2, 128), nn.ReLU(), nn.Linear(128, 128), nn.ReLU(), nn.Linear(128, 50)) for _ in range(K)]
    W = {}
    for name, idx in (("1", 0), ("2", 2), ("3", 4)):
        W["W" + name] = torch.stack([n_[idx].weight.detach() for n_ in nets]).numpy()
        W["b" + name] = torch.stack([n_[idx].bias.detach() for n_ in nets]).numpy()
    basis, _ = vlg.construct_nullspace_basis(n_poly)
    g = dict(a=(torch.rand(N, 2) * 6 - 3).numpy(), b=(torch.rand(N, 2) * 6 - 3).numpy(),
             omega_init=(0.1 * torch.randn(N, n_poly + 1, 2)).numpy(), basis=basis.numpy(), n_poly=n_poly, **W)
    dec = make_decoders(vlg, g, K)
    t = torch.linspace(0, 1, T, device="cuda")
    seed, id0 = 99, 7
    draws = np.stack([O.counter_draws(seed, np.arange(N) + id0, s_, T, M, K) for s_ in range(S)])
    r = O.optimize_steps(g["a"].astype(np.float64), g["b"].astype(np.float64), g["omega_init"].astype(np.float64),
                         g["basis"].astype(np.float64), Hh.tgrid(T, np.float64), n_poly, Hh.decoder_list(W, K, np.float64), draws, S)
    out, fill = {}, {}
    for prec in ("fp32", "tf32", "f16", "f16x3", "f16x3f"):
        model = make_model(vlg, g)
        st = {}
        _, trace = vlg.optimize_splines(model, dec, t, S, M=M, seed=seed, curve_id0=id0, precision=prec, return_trace=True,
                                        stats=st if prec != "fp32" else None)
        out[prec] = (trace.cpu().numpy(), model.omega.cpu().numpy())
        if st:
            fill[prec] = st["rows"] / (128.0 * st["items"])
    assert np.abs(out["fp32"][0] / r["energy"] - 1).max() < 1e-5
    assert np.abs(out["fp32"][1] - r["omega"]).max() < 5e-6
    for tc in ("tf32", "f16"):
        assert np.abs(np.sqrt(out[tc][0] / r["energy"]) - 1).max() < 5e-3   # random-init nets: smooth, small energies
        assert np.abs(out[tc][1] - r["omega"]).max() < 0.25 * S * 1e-3 + 1e-6
    assert np.abs(out["f16x3"][0] / r["energy"] - 1).max() < 1e-4              # the 3-term split meets the fp32 bound
    assert np.abs(out["f16x3"][1] - r["omega"]).max() < 2e-5
    assert np.abs(out["f16x3f"][0][0] / r["energy"][0] - 1).max() < 1e-4       # default arithmetic: the energy of a given curve is fp32-grade,
    assert np.abs(out["f16x3f"][0] / r["energy"] - 1).max() < 1e-3             # later steps see the 11-bit gradient operands
    assert np.abs(out["f16x3f"][1] - r["omega"]).max() < 0.25 * S * 1e-3 + 1e-6
    # multi-curve windows: several whole curves share a window, so one decoder's rows fill its 128-row items
    # (a 256-point curve alone would leave them ~12 % full)
    print("item fill:", fill)
    assert all(f > 0.6 for f in fill.values()), fill


@pytest.mark.parametrize("tc", ["f16", "f16x3", "f16x3f", "tf32"])
def test_multi_curve_windows_are_shard_independent(vlg, tc):
    """K = 64, T = 256: windows hold several whole curves, so WHICH curves share a window depends on where a
    shard starts.  Each (point, decoder) row's dz goes to its own draw-slot cell and the cells of a point are added in
    slot order: results are bit-identical for any grouping -- full launch, shards of odd sizes, repeated runs --
    and match the one-curve-per-launch result (N = 1 launches cannot share windows)."""
    rng = np.random.default_rng(3)
    K, T, N, S, n_poly = 64, 256, 23, 2, 8
    W = dict(W1=rng.normal(size=(K, 128, 2)) * 0.7, b1=rng.normal(size=(K, 128)) * 0.3,
             W2=rng.normal(size=(K, 128, 128)) * 0.09, b2=rng.normal(size=(K, 128)) * 0.1,
             W3=rng.normal(size=(K, 50, 128)) * 0.09, b3=rng.normal(size=(K, 50)) * 0.1)
    dec = make_decoders(vlg, {k: v.astype(np.float32) for k, v in W.items()}, K)
    basis, _ = vlg.construct_nullspace_basis(n_poly)
    a = torch.tensor(rng.uniform(-3, 3, (N, 2)), dtype=torch.float32)
    b = torch.tensor(rng.uniform(-3, 3, (N, 2)), dtype=torch.float32)
    om = torch.tensor(0.1 * rng.normal(size=(N, n_poly + 1, 2)), dtype=torch.float32)
    t = torch.linspace(0, 1, T, device="cuda")

    def run(lo, hi):
        m = vlg.GeodesicSplineBatch(a[lo:hi].cuda(), b[lo:hi].cuda(), basis.cuda(), om[lo:hi].cuda(), n_poly)
        e = vlg.optimize_splines(m, dec, t, S, M=2, seed=9, curve_id0=lo, precision=tc)
        return m.omega.clone(), e.clone()

    ref_om, ref_e = run(0, N)
    assert bool(torch.isfinite(ref_e).all())
    o2, e2 = run(0, N)
    assert torch.equal(o2, ref_om) and torch.equal(e2, ref_e)
    for cuts in ([0, 5, 12, 23], [0, 1, 2, 9, 10, 23]):
        oms, es = zip(*[run(lo, hi) for lo, hi in zip(cuts[:-1], cuts[1:])])
        assert torch.equal(torch.cat(oms), ref_om) and torch.equal(torch.cat(es), ref_e)


@pytest.mark.parametrize("prec,tol", [("fp32", 1e-3), ("tf32", 1e-3), ("f16", 1e-3), ("f16x3", 1e-3)])
def test_full_config1_1000_steps_final_lengths(vlg, prec, tol):
    """North-star statement: BASELINE config 1 at full length (45 curves, K=10, M=2, T=2000, 1000 Adam
    steps) against the reference's own fp64 run with the same counter-based draws
    (tests/golden/make_golden_full1000.py).  Free-running, so this bounds the accumulated drift of the
    whole trajectory, not one step."""
    path = Hh.GOLDEN / "ens_seed12_full1000.npz"
    if not path.exists():
        pytest.skip("golden not generated (tests/golden/make_golden_full1000.py, ~1 h of CPU)")
    g = dict(np.load(path))
    s = Hh.load("splines_seed12_euclidean_10")
    inp = dict(a=s["a"], b=s["b"], omega_init=s["omega_init"], basis=s["basis"], n_poly=int(s["n_poly"]))
    model = make_model(vlg, inp)
    dec = make_decoders(vlg, Hh.load("evae_seed12_decoders"), 10)
    t = torch.linspace(0, 1, 2000, device="cuda")
    steps = int(g["steps"])
    _, trace = vlg.optimize_splines(model, dec, t, steps, M=2, seed=int(g["seed"]), curve_id0=0, precision=prec,
                                    return_trace=True)
    trace = trace.cpu().numpy()
    for i, st in enumerate(g["energy_steps"]):
        rel = np.abs(np.sqrt(trace[int(st)] / g["energy_f64"][i]) - 1).max()
        print(f"{prec}: step {int(st):4d} max rel length err vs reference fp64 = {rel:.2e}")
    final = np.abs(np.sqrt(trace[-1]) / g["final_length_f64"] - 1).max()
    assert final < tol, final
    assert np.abs(model.omega.cpu().numpy() - g["omega_f64"]).max() < 5e-2


@pytest.mark.parametrize("prec", ["f16", "f16x3", "f16x3f", "tf32"])
def test_full_pair_list_sharding_and_modes_agree(vlg, prec):
    """BASELINE config 3 at its full width (8778 pairs, K=10, M=2, T=2000), size-independent properties:
    the 8-way shard of the pair list reproduces the single-launch result bit for bit (the work queue hands
    curves to CTAs in a different order), every energy is finite and positive, and the two fp16 modes agree
    with each other to the single-term tolerance."""
    import bench
    w, a, b, omega, _ = bench.synthetic_workload(bench.N_CURVES)
    dev = "cuda"
    dec = vlg.DecoderEnsemble.from_arrays(*[w[k] for k in ("W1", "b1", "W2", "b2", "W3", "b3")], dev)
    basis, _ = vlg.construct_nullspace_basis(4)
    t = torch.linspace(0, 1, 2000, device=dev)
    N, S = bench.N_CURVES, 3

    def run(lo, hi, p):
        m = vlg.GeodesicSplineBatch(a[lo:hi].to(dev), b[lo:hi].to(dev), basis.to(dev), omega[lo:hi].to(dev), 4)
        e = vlg.optimize_splines(m, dec, t, S, M=2, seed=4, curve_id0=lo, precision=p)
        return m.omega, e

    om_full, e_full = run(0, N, prec)
    assert bool(torch.isfinite(e_full).all()) and float(e_full.min()) > 0
    from vlg_b200.sharding import shard_range
    oms, es = zip(*[run(*shard_range(N, r, 8), prec) for r in range(8)])
    assert torch.equal(torch.cat(oms), om_full) and torch.equal(torch.cat(es), e_full)
    if prec == "f16":
        _, e_x3 = run(0, N, "f16x3")
        assert float((torch.sqrt(e_full / e_x3) - 1).abs().max()) < 2e-3


@pytest.mark.parametrize("prec", ["fp32", "tf32", "f16", "f16x3", "f16x3f"])
@pytest.mark.parametrize("T,N,K,M,n_poly", [(513, 150, 7, 2, 4), (2000, 5, 10, 2, 4), (130, 3, 3, 1, 8), (256, 20, 70, 3, 8)])
def test_kernels_write_only_inside_their_buffers(vlg, prec, T, N, K, M, n_poly):
    """Guard bands: the workspace is handed over at exactly vlg_workspace_bytes, and it, the curve state and
    the outputs sit inside larger buffers filled with a pattern; nothing outside the declared extents may
    change (compute-sanitizer is not available on the GPU pool, this is the bounds check we can run)."""
    from vlg_b200 import ops
    rng = np.random.default_rng(T + K)
    W = dict(W1=rng.normal(size=(K, 128, 2)) * 0.7, b1=rng.normal(size=(K, 128)) * 0.3,
             W2=rng.normal(size=(K, 128, 128)) * 0.09, b2=rng.normal(size=(K, 128)) * 0.1,
             W3=rng.normal(size=(K, 50, 128)) * 0.09, b3=rng.normal(size=(K, 50)) * 0.1)
    g = {k: v.astype(np.float32) for k, v in W.items()}
    dec = make_decoders(vlg, g, K)
    basis, _ = vlg.construct_nullspace_basis(n_poly)
    dev, G, S, Kb = "cuda", 4096, 2, n_poly + 1
    code = ops.PRECISIONS[prec]

    def guarded(nbytes_or_tensor, dtype=torch.float32):
        """-> (view of the payload, full byte buffer, payload byte range)"""
        if isinstance(nbytes_or_tensor, int):
            nbytes, src = nbytes_or_tensor, None
        else:
            src = nbytes_or_tensor.contiguous()
            nbytes = src.numel() * src.element_size()
        nbytes_al = (nbytes + 255) // 256 * 256
        buf = torch.full((G + nbytes_al + G,), 0xA5, dtype=torch.uint8, device=dev)
        view = buf[G:G + nbytes].view(dtype) if dtype != torch.uint8 else buf[G:G + nbytes]
        if src is not None:
            view.copy_(src.to(dev).view(-1))
        return view, buf, (G, G + nbytes)

    omega0 = torch.tensor(0.1 * rng.normal(size=(N, Kb, 2)), dtype=torch.float32)
    om, om_buf, om_rng = guarded(omega0)
    m_, m_buf, m_rng = guarded(torch.zeros(N, Kb, 2))
    v_, v_buf, v_rng = guarded(torch.zeros(N, Kb, 2))
    e_, e_buf, e_rng = guarded(torch.zeros(N))
    tr, tr_buf, tr_rng = guarded(torch.zeros(S, N))
    nws = ops.workspace_bytes(N, T, n_poly, K, M, code)
    ws, ws_buf, ws_rng = guarded(int(nws), torch.uint8)
    a = torch.tensor(rng.uniform(-3, 3, (N, 2)), dtype=torch.float32, device=dev)
    b = torch.tensor(rng.uniform(-3, 3, (N, 2)), dtype=torch.float32, device=dev)
    t = torch.linspace(0, 1, T, device=dev)
    ops.optimize_steps(dec.packed, dec.K, dec.X, K, n_poly, M, S, 0, a, b, om.view(N, Kb, 2), m_.view(N, Kb, 2), v_.view(N, Kb, 2),
                       basis.to(dev).float().contiguous(), t, None, None, 3, 11, 1e-3, 0.9, 0.999, 1e-8, 1000.0, e_, tr.view(S, N), code,
                       ws if nws else None)
    torch.cuda.synchronize()
    for name, buf, (lo, hi) in (("omega", om_buf, om_rng), ("adam_m", m_buf, m_rng), ("adam_v", v_buf, v_rng),
                                ("energy", e_buf, e_rng), ("trace", tr_buf, tr_rng), ("workspace", ws_buf, ws_rng)):
        assert bool((buf[:lo] == 0xA5).all()), f"{name}: write below the buffer"
        assert bool((buf[hi:] == 0xA5).all()), f"{name}: write above the buffer"
    assert bool(torch.isfinite(e_).all()) and not torch.equal(om.view(N, Kb, 2).cpu(), omega0)


# ---------------------------------------------------------------------------------------------
# The BENCHMARKED job against the reference: curves of bench.synthetic_workload (BASELINE config 3), 1000
# free-running Adam steps, final geodesic length sqrt(E) against the reference's own loop in fp64 -- with the
# reference's own fp32-vs-fp64 gap on the same curve beside it (tests/golden/make_golden_config3.py).
# ---------------------------------------------------------------------------------------------
def _run_config3_curves(vlg, ids, prec, steps=1000):
    import bench
    w, a, b, omega, _ = bench.synthetic_workload(bench.N_CURVES)
    dev = "cuda"
    dec = vlg.DecoderEnsemble.from_arrays(*[w[k] for k in Hh.DEC_KEYS], dev)
    basis, _ = vlg.construct_nullspace_basis(4)
    t = torch.linspace(0, 1, 2000, device=dev)
    out = np.zeros(len(ids))
    # contiguous runs of global curve ids share a launch (the draws are keyed on the global id)
    runs, start = [], 0
    for i in range(1, len(ids) + 1):
        if i == len(ids) or ids[i] != ids[i - 1] + 1:
            runs.append((start, i))
            start = i
    for lo, hi in runs:
        sel = torch.as_tensor(ids[lo:hi])
        m = vlg.GeodesicSplineBatch(a[sel].to(dev), b[sel].to(dev), basis.to(dev), omega[sel].to(dev), 4)
        done = 0
        while done < steps:
            e = vlg.optimize_splines(m, dec, t, min(100, steps - done), M=2, seed=0, curve_id0=int(ids[lo]), precision=prec)
            done += 100
        out[lo:hi] = np.sqrt(e.cpu().numpy().astype(np.float64))
    return out


@pytest.mark.parametrize("prec", ["fp32", "f16x3", "f16x3f", "f16", "tf32"])
def test_config3_final_lengths_against_reference_fp64(vlg, prec):
    """north_star: <= 1e-3 relative final geodesic length.  The golden holds 64 curves of the benchmarked job after
    1000 free-running Adam steps of the reference's own loop in fp64 and in fp32: the first 49 curves (an unselected
    sample) and the 15 curves of all 8778 on which the arithmetic modes diverged most in a full GPU run.  Adam
    normalises the gradient, so rounding-level differences are amplified along badly conditioned curves: the
    reference's OWN fp32 run is within 1.0e-4 of its fp64 run on the unselected curves but off by up to 1.05e-2
    (7 of 15 beyond 1e-3) on the selected ones.  Hence:
      * every mode meets 1e-3 on the unselected sample (2e-3 worst case allowed for the 11-bit modes, which sit at
        8e-4 / 9.5e-4 there);
      * the fp32-grade modes (fp32 kernel, 3-term tensor-core split) are statistically the reference's own fp32:
        median <= 1e-5, no more curves beyond 1e-3 than the reference's fp32 has (+2), worst curve <= 2x its worst;
      * the default arithmetic (f16x3f: 3-term forward GEMMs, single-term backward GEMMs) meets the same outlier
        bars and 1e-3 on the unselected sample (measured 1.3e-4, the reference's own fp32: 1.0e-4), median <= 5e-5;
      * the single-term modes (fp16 / TF32 operands: 2.5e-4 per step) stay within 2 % everywhere, median <= 5e-4.
    The table is printed."""
    g = Hh.load("config3_synth_1000")
    ids = g["ids"].astype(np.int64)
    ref = g["final_length_f64"]
    gap = np.abs(g["final_length_f32"].astype(np.float64) / ref - 1)
    got = _run_config3_curves(vlg, ids, prec, int(g["steps"]))
    err = np.abs(got / ref - 1)
    plain = np.arange(len(ids)) < 49          # ids 0..48: not selected for anything
    order = np.argsort(-err)
    print(f"\n[{prec}] final length vs reference fp64: unselected 49 curves: median {np.median(err[plain]):.1e} max {err[plain].max():.1e} "
          f"(reference fp32: median {np.median(gap[plain]):.1e} max {gap[plain].max():.1e}); 15 worst-diverging: median "
          f"{np.median(err[~plain]):.1e} max {err[~plain].max():.1e}, {int((err[~plain] > 1e-3).sum())} beyond 1e-3 "
          f"(reference fp32: median {np.median(gap[~plain]):.1e} max {gap[~plain].max():.1e}, {int((gap[~plain] > 1e-3).sum())} beyond 1e-3)")
    for i in order[:6]:
        print(f"   curve {ids[i]:5d}: err {err[i]:.2e}   reference fp32-vs-fp64 gap {gap[i]:.2e}")
    err32 = np.abs(got / g["final_length_f32"].astype(np.float64) - 1)
    print(f"   against the reference's fp32 run: median {np.median(err32):.1e}, unselected max {err32[plain].max():.1e}, overall max {err32.max():.1e}")
    assert np.isfinite(got).all()
    if prec in ("fp32", "f16x3", "f16x3f"):
        # (f16x3f: energies fp32-grade, gradient GEMMs on 11-bit operands -- the trajectories differ a little more)
        assert err[plain].max() <= 1e-3 and np.median(err) <= (5e-5 if prec == "f16x3f" else 1e-5)
        assert (err > 1e-3).sum() <= (gap > 1e-3).sum() + 2
        assert err.max() <= 2 * gap.max()
    else:
        assert np.quantile(err[plain], 0.9) <= 1e-3 and err[plain].max() <= 2e-3
        assert err.max() <= 2e-2 and np.median(err) <= 5e-4
