"""Cost of the differentiable energy on the config-3 workload (bench.synthetic_workload, default precision):
(a) forward-only compute_energy_mc, (b) compute_energy_mc with grad + .backward(), (c) optimize_splines(steps=1).
CUDA events, L2 flushed (256 MiB write) before every timed call as bench.py does, the three alternated; prints the
median of the runs per measurement, with the card name and power limit read in the same run.

    python scratch/energy_grad_rate.py [--runs 7]
"""
import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import bench  # noqa: E402
import vlg_b200  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=7)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a B200"
    dev = "cuda"
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()[0]
    w, a, b, omega, _ = bench.synthetic_workload(bench.N_CURVES)
    dec = vlg_b200.DecoderEnsemble.from_arrays(*[w[k] for k in ("W1", "b1", "W2", "b2", "W3", "b3")], dev)
    basis = vlg_b200.construct_nullspace_basis(bench.N_POLY)[0]
    t = torch.linspace(0, 1, bench.T_POINTS, device=dev)
    M = bench.M_MC
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def model(grad):
        m = vlg_b200.GeodesicSplineBatch(a.to(dev), b.to(dev), basis.to(dev), omega.to(dev), bench.N_POLY)
        m.omega.requires_grad_(grad)
        return m

    m_fwd, m_grad, m_opt = model(False), model(True), model(False)

    def fwd():
        vlg_b200.compute_energy_mc(m_fwd, dec, t, M, precision=None, check=False)

    def grad():
        m_grad.omega.grad = None
        vlg_b200.compute_energy_mc(m_grad, dec, t, M, precision=None, check=False).sum().backward()

    def opt():
        vlg_b200.optimize_splines(m_opt, dec, t, 1, M=M, check=False)

    legs = {"a_forward": fwd, "b_grad_backward": grad, "c_optimize_1step": opt}
    times = {k: [] for k in legs}
    for fn in legs.values():   # warm-up: module load, first launches
        fn()
        fn()
    torch.cuda.synchronize()
    for r in range(args.runs):
        for name, fn in legs.items():
            flush.fill_(r & 0xFF)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1))
    med = {k: statistics.median(v) for k, v in times.items()}
    print(json.dumps({"card": card, "N": bench.N_CURVES, "T": bench.T_POINTS, "K": bench.K_DEC, "M": M,
                      "precision": vlg_b200.DEFAULT_PRECISION, "runs": args.runs,
                      "median_ms": {k: round(v, 3) for k, v in med.items()},
                      "spread_ms": {k: round(max(v) - min(v), 3) for k, v in times.items()},
                      "b_over_a": round(med["b_grad_backward"] / med["a_forward"], 3),
                      "b_over_c": round(med["b_grad_backward"] / med["c_optimize_1step"], 3)}))


if __name__ == "__main__":
    main()
