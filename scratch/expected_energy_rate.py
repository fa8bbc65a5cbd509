"""Time and peak memory of the expected ensemble energy (expected_curve_energy) against the MC energy and against the
same closed form written in plain torch on decoders(z).

Shapes: BASELINE config 3 (8778 curves, T = 2000, the committed eVAE seed-12 decoders, K = 10, X = 50) and config 5
(100 000 curves, T = 256, K = 64 random-init decoders), with the curves bench.py builds (imported, not copied).
Paths, each forward only (no_grad) and forward + .backward() to omega:
  expected_curve_energy(decoders, model(t_vals))          in f16x3f, f16x3 and (config 3) fp32
  compute_energy_mc(model, decoders, t_vals, M=2)         the fused MC energy (default precision)
  the closed form in plain torch on decoders(model(t_vals)), in curve chunks that fit (default precision)
CUDA events around each call (it ends in a synchronise), median of --runs runs with the paths alternated, after one
warm-up call of every path; torch.cuda.max_memory_allocated of each path (over its runs, reset before each call).
Prints the card name and power limit of the same run.

    python scratch/expected_energy_rate.py [--runs 5] [--configs 3 5]
"""
import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402
import vlg_b200  # noqa: E402


def torch_expected_energy(decoders, z, chunk):
    """sum_s ||mu_{s+1} - mu_s||^2 + sum_t c_t V_t on decoders(z) [K, T, n, X], n curves at a time."""
    T = z.shape[0]
    c = torch.full((T, 1), 2.0, device=z.device)
    c[0] = c[-1] = 1.0
    out = []
    for n0 in range(0, z.shape[1], chunk):
        x = decoders(z[:, n0:n0 + chunk])
        mu = x.mean(0)
        V = ((x - mu) ** 2).sum(-1).mean(0)
        out.append(((mu[1:] - mu[:-1]) ** 2).sum(-1).sum(0) + (c * V).sum(0))
    return torch.cat(out)


def torch_expected_energy_backward(decoders, z, chunk):
    """The same with dE/dz formed chunk by chunk (each chunk's graph freed by its own backward), then carried to the
    spline parameters by one z.backward: the plain-torch path that fits in memory."""
    dz, out = [], []
    for n0 in range(0, z.shape[1], chunk):
        zc = z[:, n0:n0 + chunk].detach().requires_grad_(True)
        e = torch_expected_energy(decoders, zc, zc.shape[1])
        e.sum().backward()
        dz.append(zc.grad)
        out.append(e.detach())
    z.backward(torch.cat(dz, 1))
    return torch.cat(out)


def run_config(cfg_id, runs):
    cfg = bench.make_config(cfg_id)
    dev = "cuda"
    N, T, n_poly = cfg["N"], cfg["T"], cfg["n_poly"]
    w = cfg["w"]
    ens = vlg_b200.DecoderEnsemble.from_arrays(*[np.asarray(w[k], dtype=np.float32) for k in ("W1", "b1", "W2", "b2", "W3", "b3")], dev)
    basis, _ = vlg_b200.construct_nullspace_basis(n_poly, dev)
    t = torch.linspace(0, 1, T, device=dev)
    X = ens.X
    chunk = max(1, int(2.5e9 // (4 * len(ens) * T * X)))   # [K, T, chunk, X] fp32 of about 2.5 GB

    def model(grad):
        m = vlg_b200.GeodesicSplineBatch(cfg["a"].to(dev), cfg["b"].to(dev), basis, cfg["omega"].to(dev), n_poly)
        m.omega.requires_grad_(grad)
        return m

    def ee(prec, grad):
        def f():
            m = model(grad)
            if grad:
                vlg_b200.expected_curve_energy(ens, m(t), precision=prec).sum().backward()
            else:
                with torch.no_grad():
                    vlg_b200.expected_curve_energy(ens, m(t), precision=prec)
        return f

    def mc(grad):
        def f():
            m = model(grad)
            if grad:
                vlg_b200.compute_energy_mc(m, ens, t, 2, precision=None).sum().backward()
            else:
                with torch.no_grad():
                    vlg_b200.compute_energy_mc(m, ens, t, 2, precision=None)
        return f

    def plain(grad):
        def f():
            m = model(grad)
            if grad:
                torch_expected_energy_backward(ens, m(t), chunk)
            else:
                with torch.no_grad():
                    torch_expected_energy(ens, m(t), chunk)
        return f

    precs = ["f16x3f", "f16x3"] + (["fp32"] if cfg_id == 3 else [])
    paths = {}
    for grad in (False, True):
        tag = "fwd+bwd" if grad else "fwd"
        for p in precs:
            paths[f"expected {p} {tag}"] = ee(p, grad)
        paths[f"compute_energy_mc M=2 {tag}"] = mc(grad)
        paths[f"plain torch on decoders(z) {tag}"] = plain(grad)

    # agreement of the three energies on this workload (f16x3 expected energy as the yardstick)
    with torch.no_grad():
        m = model(False)
        e_x = vlg_b200.expected_curve_energy(ens, m(t), precision="f16x3")
        e_t = torch_expected_energy(ens, m(t), chunk)
        e_mc = vlg_b200.compute_energy_mc(m, ens, t, 2, precision=None)
    agree = {"plain_torch_vs_expected_max_rel": float(((e_t - e_x).abs() / e_x.abs()).max()),
             "mc_M2_vs_expected_median_rel": float(((e_mc - e_x).abs() / e_x.abs()).median()),
             "mc_M2_vs_expected_max_rel": float(((e_mc - e_x).abs() / e_x.abs()).max())}
    del e_x, e_t, e_mc, m

    times = {k: [] for k in paths}
    peak = {k: 0 for k in paths}
    for f in paths.values():
        f()
    torch.cuda.synchronize()
    for _ in range(runs):
        for k, f in paths.items():
            torch.cuda.empty_cache()
            torch.cuda.reset_peak_memory_stats()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) * 1e-3)
            peak[k] = max(peak[k], torch.cuda.max_memory_allocated())
    res = {"config": cfg["name"], "N": N, "T": T, "K": len(ens), "X": X, "weights": cfg["weights"],
           "plain_torch_chunk_curves": chunk, "runs": runs, "agreement": agree}
    for k in paths:
        res[k] = {"ms_median": round(statistics.median(times[k]) * 1e3, 2),
                  "ms_min": round(min(times[k]) * 1e3, 2), "ms_max": round(max(times[k]) * 1e3, 2),
                  "peak_GB": round(peak[k] / 1e9, 3)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--configs", type=int, nargs="+", default=[3, 5])
    ap.add_argument("--out", default=None, help="also write the JSON here")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a B200"
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()[0]
    out = {"card": card, "results": [run_config(c, args.runs) for c in args.configs]}
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        Path(args.out).write_text(text)


if __name__ == "__main__":
    main()
