#!/usr/bin/env python
"""Benchmark of the geodesic curve-energy hot path (BASELINE.json metric: spline-steps/sec,
8778-pair 10-decoder eVAE energy optimisation).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--precision f16|f16x3|tf32|fp32]
                    [--config 3|5|2] [--dump-outputs DIR]

A "step" is one Adam step of EVERY curve of the workload (= n_curves spline-steps): spline
evaluation, all-decoder forward + input-gradient backward, MC pair energy, Adam -- one pass of
the hot path over the whole pair list.  For N > 1 (torchrun, one rank per GPU) the pair list is
split into contiguous shards, no collective on the step path (strong scaling of the named job);
the one exchange -- the final gather of omega / lengths on rank 0 -- is inside the e2e leg.

One JSON line on stdout (rank 0):
  value      device-resident throughput of the headline arithmetic (vlg_b200.DEFAULT_PRECISION)
  e2e        the same metric through the public API with HOST buffers: H2D of the curve state,
             the launch, (N > 1: gather on rank 0,) D2H of omega + energies, inside the timed region
  roofline   algorithmic tensor FLOP/s of the step kernel against the measured dense bf16 peak, plus
             the tensor FLOP/s the kernel really executed (row compaction skips unselected decoders)
             and the tensor-pipe utilisation
  other_modes  the other arithmetic modes on the same workload (secondary entries)
  cpu_baseline / gpu_eager_baseline  the reference's own loop (oracle/_ref: unmodified reference
             modules) on this box's host cores and, eager fp32, on the same GPU -- bounded samples
`--impl reference` prints the CPU arm alone.  Workloads: --config 3 (default, the headline),
--config 5 (100k pairs, 64 decoders, n_poly 8, T=256), --config 2 (single decoder, 8778 splines).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

N_CURVES = 8778          # 133 classes -> 133*132/2 pairs (BASELINE config 3)
T_POINTS = 2000          # src/optimize.py:130
N_POLY = 4
K_DEC = 10
M_MC = 2
FLOP_PER_POINT_DECODER = 92160  # fwd + input-grad bwd of 2->128->128->50 (SURVEY §8d)
# tensor FLOPs of ONE executed 128-row item (four GEMMs: 128x128x128, 128x64x128, 128x128x64, 128x128x128)
FLOP_PER_ITEM = 2 * 128 * (128 * 128 + 64 * 128 + 128 * 64 + 128 * 128)
MMAS_PER_ITEM = {"f16": 28, "f16x3": 84, "f16x3f": 60, "tf32": 56}   # M=128 instructions; 63-69 cycles each (DESIGN.md §4.4)
MMA_TERMS = {"f16": 1, "f16x3": 3, "f16x3f": 60.0 / 28.0, "tf32": 1}
METRIC = "spline-steps/sec, 8778-pair 10-decoder eVAE energy opt"
# arithmetic of the two 128-wide decoder layers (layer 1, the energy, the spline and Adam are fp32 everywhere)
PRECISION_NOTE = {
    "f16": "f16: tcgen05 kind::f16, fp16 operands (11-bit significand, as TF32), fp32 accumulate; <=1e-3 rel. on lengths",
    "f16x3": "f16x3: tcgen05 kind::f16, hi+lo fp16 operands, 3 MMAs per product, fp32 accumulate; fp32-grade (2e-6 rel. per-step energy)",
    "f16x3f": "f16x3f: f16x3 in the forward GEMMs (energies fp32-grade), single-term fp16 operands in the backward GEMMs",
    "tf32": "tf32: tcgen05 kind::tf32, fp32 accumulate; <=1e-3 rel. on lengths",
    "fp32": "fp32: CUDA-core FFMA; <=1e-4 rel. per-step energy",
}
KERNEL_NAME = {"f16": "tc_curve_kernel<true, FMT_F16>", "f16x3": "tc_curve_kernel<true, FMT_F16X3>",
               "f16x3f": "tc_curve_kernel<true, FMT_F16X3F>",
               "tf32": "tc_curve_kernel<true, FMT_TF32>", "fp32": "simt_curve_kernel<true>"}
DTYPE = {"f16": "f16", "f16x3": "f16x3", "f16x3f": "f16x3f", "tf32": "tf32", "fp32": "f32"}


# ----------------------------------------------------------------------------------------------
# workloads
# ----------------------------------------------------------------------------------------------

def random_decoders(K, seed=0):
    """default nn.Linear init, 2 -> 128 -> 128 -> 50, K decoders (src/train.py:80-85)."""
    import torch.nn as nn
    torch.manual_seed(seed)
    nets = [nn.Sequential(nn.Linear(2, 128), nn.ReLU(), nn.Linear(128, 128), nn.ReLU(), nn.Linear(128, 50))
            for _ in range(K)]
    w = {}
    for name, idx in (("1", 0), ("2", 2), ("3", 4)):
        w["W" + name] = torch.stack([n[idx].weight.detach() for n in nets]).numpy()
        w["b" + name] = torch.stack([n[idx].bias.detach() for n in nets]).numpy()
    return w


def synthetic_workload(n_curves, seed=0):
    """tasic-pca50-shaped synthetic job (BASELINE config 3): the committed eVAE seed-12 decoder weights when
    the golden file is present (else default nn.Linear init), random end points in the latent box,
    near-straight initial splines (the 'euclidean' init is ~0)."""
    gold = ROOT / "tests" / "golden" / "evae_seed12_decoders.npz"
    if gold.exists():
        w = dict(np.load(gold))
        weights = "evae_seed12 checkpoint decoders"
    else:
        w = random_decoders(K_DEC, seed)
        weights = "random-init decoders"
    g = torch.Generator().manual_seed(seed)
    a = torch.rand(n_curves, 2, generator=g) * 7 - 3.5
    b = torch.rand(n_curves, 2, generator=g) * 7 - 3.5
    omega = 0.05 * torch.randn(n_curves, N_POLY + 1, 2, generator=g)
    return w, a, b, omega, weights


def make_config(cfg: int):
    """-> dict(name, N, T, K, M, n_poly, w, a, b, omega, weights) for a BASELINE.json configuration."""
    if cfg == 3:
        w, a, b, omega, weights = synthetic_workload(N_CURVES)
        return dict(name="BASELINE config 3: 8778 pairs (133 classes), 10-decoder eVAE, T=2000, n_poly=4, M=2",
                    N=N_CURVES, T=T_POINTS, K=K_DEC, M=M_MC, n_poly=N_POLY, w=w, a=a, b=b, omega=omega, weights=weights)
    if cfg == 5:   # SURVEY §8d row 5
        N, K, n_poly, T = 100_000, 64, 8, 256
        w = random_decoders(K, 0)
        g = torch.Generator().manual_seed(0)
        a = torch.rand(N, 2, generator=g) * 6 - 3
        b = torch.rand(N, 2, generator=g) * 6 - 3
        omega = 0.1 * torch.randn(N, n_poly + 1, 2, generator=g)
        return dict(name="BASELINE config 5: 100k pairs, 64-decoder ensemble, n_poly=8, T=256, M=2, random-init weights",
                    N=N, T=T, K=K, M=2, n_poly=n_poly, w=w, a=a, b=b, omega=omega, weights="random-init decoders (torch seed 0)")
    if cfg == 2:   # single-decoder VAE, all 133-class pairs; deterministic energy (K=1, M=1)
        gold = ROOT / "tests" / "golden" / "single_seed123.npz"
        if gold.exists():
            g_ = np.load(gold)
            w = {k: g_[k] for k in ("W1", "b1", "W2", "b2", "W3", "b3")}
            weights = "vae_best_seed123 decoder (rows 0:50 of the last layer)"
        else:
            w, weights = random_decoders(1, 0), "random-init decoder"
        _, a, b, omega, _ = synthetic_workload(N_CURVES)
        return dict(name="BASELINE config 2: single-decoder VAE, 8778 splines, T=2000, n_poly=4 (deterministic energy)",
                    N=N_CURVES, T=T_POINTS, K=1, M=1, n_poly=N_POLY, w=w, a=a, b=b, omega=omega, weights=weights)
    raise SystemExit(f"unknown --config {cfg}")


def shard_range(n, rank, world):
    from vlg_b200.sharding import shard_range as sr
    return sr(n, rank, world)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peak():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        d = json.loads(f.read_text())
        return float(d["bf16_tflops_sustained"]), "MEASURED_PEAKS.json bf16_tflops_sustained (dense bf16; TF32 tensor rate is half)"
    return 1400.0, "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------
# Reference arms: the reference's OWN loop (src/optimize.py:152-162 of the reference, unmodified
# modules from oracle/_ref -- see oracle/make_ref.py), on the host cores or eager on the GPU.
# Falls back to the oracle's PyTorch port (oracle/torch_port.py) when oracle/_ref is absent.
# ----------------------------------------------------------------------------------------------

def _reference_modules():
    try:
        from oracle import make_ref
        if not make_ref.available():
            make_ref.make(verbose=False)     # only possible where /root/reference is mounted
        if make_ref.available():
            return make_ref.import_reference()
    except Exception as exc:  # noqa: BLE001 - any failure -> port
        print(f"[bench] oracle/_ref unavailable ({exc}); using the oracle port", file=sys.stderr)
    return None


def reference_loop_rate(cfg, device, steps, warmup, sample, threads=None):
    """spline-steps/s of the reference loop on `device` for the first `sample` curves of the workload
    (reference batch-size is 200; steps are homogeneous).  Returns (rate, kind, sample description)."""
    import vlg_b200
    w, K, M, T, n_poly = cfg["w"], cfg["K"], cfg["M"], cfg["T"], cfg["n_poly"]
    dev = torch.device(device)
    if dev.type == "cpu":
        torch.set_num_threads(threads or os.cpu_count() or 1)
    basis = vlg_b200.construct_nullspace_basis(n_poly)[0].to(dev)
    t = torch.linspace(0, 1, T, device=dev)
    a, b, om = (cfg[k][:sample].clone().to(dev) for k in ("a", "b", "omega"))
    mods = _reference_modules() if (K == 10 and M > 0) else None
    if mods is not None:
        ref_opt, ref_train, _ = mods
        model = ref_train.EVAE(ref_train.GaussianPrior(2), ref_train.GaussianEncoder(ref_train.make_encoder_net(50, 2)),
                               ref_train.GaussianDecoder(ref_train.make_decoder_net(2, 50)), num_decoders=K)
        with torch.no_grad():
            for i, d in enumerate(model.decoder):
                for idx, (wk, bk) in zip((0, 2, 4), (("W1", "b1"), ("W2", "b2"), ("W3", "b3"))):
                    d.decoder_net[idx].weight.copy_(torch.as_tensor(w[wk][i]))
                    d.decoder_net[idx].bias.copy_(torch.as_tensor(w[bk][i]))
        model = model.to(dev).eval()
        decoders = list(model.decoder)          # parameters keep requires_grad=True, as in src/optimize.py:103
        spl = ref_opt.GeodesicSplineBatch(a, b, basis, om, n_poly).to(dev)
        opt = torch.optim.Adam(spl.parameters(), lr=1e-3)

        def run(n):
            for _ in range(n):                   # src/optimize.py:155-162
                opt.zero_grad()
                energy = ref_opt.compute_energy_mc(spl, decoders, t, M=M)
                endpoint_error = (spl(t[-1:]) - b[None]) ** 2
                loss = energy + 1000 * endpoint_error.sum(dim=(0, 2))
                loss.sum().backward()
                opt.step()
        kind = "reference"
    else:
        from oracle import torch_port as TP
        decs = [TP.make_decoder({k: w[k][i] for k in ("W1", "b1", "W2", "b2", "W3", "b3")}).to(dev) for i in range(K)]
        m = TP.SplineBatch(a, b, basis, om, n_poly).to(dev)
        state = {"opt": None}

        def run(n):
            _, state["opt"] = TP.run_steps(m, decs, t, n, M=max(M, 1), opt=state["opt"])
        kind = "port"

    def sync():
        if dev.type == "cuda":
            torch.cuda.synchronize(dev)

    run(max(1, warmup))
    sync()
    t0 = time.perf_counter()
    run(max(1, steps))
    sync()
    dt = time.perf_counter() - t0
    what = (f"{sample} curves x {max(1, steps)} steps (T={T}, K={K}, M={M}), torch {torch.__version__} "
            + (f"CPU, {torch.get_num_threads()} threads" if dev.type == "cpu" else "CUDA eager fp32")
            + (", unmodified reference modules (oracle/_ref)" if kind == "reference" else ", oracle/torch_port.py"))
    return sample * max(1, steps) / dt, kind, what


def cpu_reference_rate(cfg, steps, warmup, budget_s):
    """CPU arm on a bounded sample: probe the per-curve-step cost, then size the sample (<= 200 curves,
    the reference's batch size) so that warm-up + timed steps take about `budget_s` seconds."""
    cores = os.cpu_count() or 1
    probe_rate, _, _ = reference_loop_rate(cfg, "cpu", 1, 1, 8, cores)
    total_steps = max(1, steps) + max(1, warmup)
    sample = int(max(4, min(200, budget_s * probe_rate / total_steps)))
    rate, kind, what = reference_loop_rate(cfg, "cpu", steps, warmup, sample, cores)
    return rate, cores, kind, what


def write_outputs(out_dir: Path, outputs):
    """<out_dir>/<name>.npy, float32 as computed, every curve: energy [N] and omega / adam_m / adam_v
    [N, n_poly + 1, 2] -- 1.1 MB for configs 2 and 3, 22 MB for config 5."""
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, x in outputs.items():
        np.save(out_dir / f"{name}.npy", x.cpu().numpy())


def workload_config(cfg, gpus, where, extra=None):
    d = {"workload": cfg["name"], "n_curves": cfg["N"], "T": cfg["T"], "K": cfg["K"], "M": cfg["M"],
         "n_poly": cfg["n_poly"], "weights": cfg["weights"],
         "sharding": f"pair list split over {gpus} GPU(s), no collective on the step path; final gather of omega/energy on rank 0 inside e2e",
         "cache": "L2 flushed (256 MiB write) between timed launches" if where == "gpu" else "n/a"}
    d.update(extra or {})
    return d


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = make_config(args.config)
    rate, cores, kind, sample = cpu_reference_rate(cfg, args.steps, args.warmup, budget_s=90.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": "spline-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * cfg["N"] / rate,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(cfg, args.gpus, "cpu", {"precision": "fp32 (PyTorch CPU)"}),
        "cpu_baseline": {"value": rate, "unit": "spline-steps/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": rate, "unit": "spline-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------

def run_gpu_arm(args):
    import torch.distributed as dist
    import vlg_b200
    from vlg_b200 import sharding

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local if world > 1 else 0)
    torch.cuda.set_device(dev)
    vlg_b200.build.build()
    precision = args.precision or vlg_b200.DEFAULT_PRECISION
    if args.config == 2 and precision in ("f16", "tf32", "f16x3f") and not args.precision:
        precision = "f16x3"     # the single-decoder drop-in's default
    if args.config == 2 and precision in ("f16", "tf32"):
        precision = "f16x3"     # 11-bit operands cannot resolve a single decoder's adjacent-point differences

    cfg = make_config(args.config)
    N, T, K, M, n_poly = cfg["N"], cfg["T"], cfg["K"], cfg["M"], cfg["n_poly"]
    w, a, b, omega = cfg["w"], cfg["a"], cfg["b"], cfg["omega"]
    lo, hi = shard_range(N, rank, world)
    n_local = hi - lo
    dec = vlg_b200.DecoderEnsemble.from_arrays(*[w[k] for k in ("W1", "b1", "W2", "b2", "W3", "b3")], dev)
    basis, _ = vlg_b200.construct_nullspace_basis(n_poly)
    basis = basis.to(dev)
    t = torch.linspace(0, 1, T, device=dev)
    # pinned host copies of this rank's shard (e2e leg) and device-resident state (value leg)
    h_a, h_b, h_om = (x[lo:hi].contiguous().pin_memory() for x in (a, b, omega))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    chunk = max(1, min(args.steps, args.chunk))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def fresh_model():
        return vlg_b200.GeodesicSplineBatch(h_a.to(dev), h_b.to(dev), basis, h_om.to(dev), n_poly)

    def timed_steps(prec, nsteps, nwarm):
        """K steps with the curve state resident in HBM; returns (ms over the region, ms inside kernels, launches,
        the launch function, what the last timed step handed back: {energy, omega, adam_m, adam_v})."""
        model = fresh_model()

        def launch(ns):
            return vlg_b200.optimize_splines(model, dec, t, ns, M=M, seed=0, curve_id0=lo, precision=prec, check=False)

        for _ in range(nwarm):
            launch(1)
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        done, events = 0, []
        while done < nsteps:
            ns = min(chunk, nsteps - done)
            flush.fill_(done & 0xFF)
            k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            k0.record()
            energy = launch(ns)
            k1.record()
            events.append((k0, k1))
            done += ns
        ev1.record()
        barrier()
        # copies: later launches (the same-load tail below) keep updating the model in place
        outputs = {"energy": energy.clone(), "omega": model.omega.clone(), "adam_m": model.adam_m.clone(),
                   "adam_v": model.adam_v.clone()}
        return ev0.elapsed_time(ev1), sum(x.elapsed_time(y) for x, y in events), len(events), launch, outputs

    # clocks are sampled (nvidia-smi, 100 ms period) from the warm-up on: the timed region of a sharded run can
    # be shorter than one sampling period, so the same load is kept up before and after it (see below)
    sampler = ClockSampler(dev.index)
    sampler.start()

    # ---- value: K steps, state resident in HBM ----
    ms_total, kernel_ms, launches, launch, outputs = timed_steps(precision, args.steps, max(args.warmup, 3))
    # untimed tail under the same load until the sampler has seen the GPU busy at least three times
    t_tail = time.time()
    while len(sampler.rows) < 3 and time.time() - t_tail < 2.0:
        launch(1)
        torch.cuda.synchronize()
    clocks = sampler.stop()
    clocks["window"] = "warm-up + timed region + same-load tail"

    # ---- e2e: same steps through the public API with host buffers (+ the final gather for N > 1) ----
    h_out_om = torch.empty((N if rank == 0 else n_local,) + tuple(h_om.shape[1:])).pin_memory()
    h_out_e = torch.empty(N if rank == 0 else n_local, dtype=torch.float32).pin_memory()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def e2e_call(ns, last):
        m2 = vlg_b200.GeodesicSplineBatch(h_a.to(dev, non_blocking=True), h_b.to(dev, non_blocking=True), basis,
                                          h_om.to(dev, non_blocking=True), n_poly)
        en = vlg_b200.optimize_splines(m2, dec, t, ns, M=M, seed=0, curve_id0=lo, precision=precision)
        if world > 1 and last:
            om_all = sharding.gather_results(m2.omega, N)       # the job's only exchange (SURVEY §8e)
            en_all = sharding.gather_results(en, N)
            if rank == 0:
                h_out_om.copy_(om_all, non_blocking=True)
                h_out_e.copy_(en_all, non_blocking=True)
        else:
            h_out_om[:n_local].copy_(m2.omega, non_blocking=True)
            h_out_e[:n_local].copy_(en, non_blocking=True)

    e2e_call(1, True)   # untimed warm-up of this path (first pinned H2D, allocator growth, NCCL gather setup)
    barrier()
    e0.record()
    done, e2e_launches = 0, 0
    while done < args.steps:
        ns = min(chunk, args.steps - done)
        e2e_call(ns, done + ns >= args.steps)
        done += ns
        e2e_launches += 1
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    h2d = (h_a.numel() + h_b.numel() + h_om.numel()) * 4
    d2h = (h_out_om.numel() + h_out_e.numel()) * 4

    # ---- executed work: one extra launch with the kernel's own counters ----
    stats = {}
    if precision != "fp32":
        vlg_b200.optimize_splines(fresh_model(), dec, t, 1, M=M, seed=0, curve_id0=lo, precision=precision, stats=stats)

    # ---- secondary entries: the other arithmetic modes on the same workload (1 GPU runs only) ----
    other = {}
    if world == 1 and not args.no_other:
        for prec in ("f16", "f16x3", "f16x3f", "tf32", "fp32"):
            if prec == precision or (K == 1 and prec in ("f16", "tf32")):
                continue
            ns = args.steps if prec != "fp32" else max(1, min(args.steps, 2))
            ms, kms, _, _, _ = timed_steps(prec, ns, 2)
            other[prec] = {"value": N * ns / (ms * 1e-3), "unit": "spline-steps/s", "steps": ns,
                           "roofline_frac": N * ns * T * K * FLOP_PER_POINT_DECODER / (kms * 1e-3) / 1e12 / measured_peak()[0],
                           "note": PRECISION_NOTE[prec]}

    if args.dump_outputs:
        outputs = {k: sharding.gather_results(v, N) for k, v in outputs.items()}
        if rank == 0:
            write_outputs(Path(args.dump_outputs), outputs)

    # max over ranks
    times = torch.tensor([ms_total, ms_e2e, kernel_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e, kernel_ms = (float(x) for x in times.cpu())

    if rank == 0:
        spline_steps = N * args.steps
        value = spline_steps / (ms_total * 1e-3)
        peak, peak_src = measured_peak()
        # roofline of the step kernel on THIS rank: algorithmic FLOPs / kernel time
        flop_per_ss = T * K * FLOP_PER_POINT_DECODER
        achieved = n_local * args.steps * flop_per_ss / (kernel_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "traffic": None, "peak_source": peak_src, "kernel": KERNEL_NAME[precision],
                "flop_per_spline_step": flop_per_ss, "kernel_ms_per_step": kernel_ms / args.steps,
                "definition": "algorithmic = the reference's dense K x T decoder evaluation (SURVEY §8d); "
                              "executed = tensor FLOPs of the 128-row items the kernel really ran (row compaction "
                              "skips decoders no segment drew; padding rows and the 3-term split are counted)"}
        if stats:
            items_per_ss = stats["items"] / n_local
            ss_per_s = n_local * args.steps / (kernel_ms * 1e-3)
            terms = MMA_TERMS[precision]
            roof["items_per_spline_step"] = items_per_ss
            roof["item_fill"] = stats["rows"] / (128.0 * max(1, stats["items"]))
            roof["executed_tflops"] = items_per_ss * FLOP_PER_ITEM * terms * ss_per_s / 1e12
            roof["executed_frac"] = roof["executed_tflops"] / peak
            sm_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6
            sms = torch.cuda.get_device_properties(dev).multi_processor_count
            roof["tensor_pipe_active_est"] = items_per_ss * MMAS_PER_ITEM[precision] * 64.0 * ss_per_s / (sm_hz * sms)
            roof["tensor_pipe_active_est_how"] = "executed MMAs x 64 cycles / (SM clock x SMs x kernel time)"
        prof = ROOT / "profiles" / "r02_ncu_metrics.json"
        if prof.exists():
            pm = json.loads(prof.read_text()).get(f"config{args.config}", {}).get(precision)
            if pm:
                roof["tensor_pipe_active"] = pm.get("sm__pipe_tc_cycles_active_pct")
                roof["ncu"] = pm
                # DRAM bytes of ONE bench launch (dram__bytes_read.sum + dram__bytes_write.sum of the same command under ncu)
                if pm.get("steps_per_launch") == chunk and pm.get("n_curves") == n_local:
                    roof["traffic"] = pm.get("dram_bytes_per_launch")
        line = {
            "metric": METRIC if args.config == 3 else f"spline-steps/sec, {cfg['name']}", "value": value,
            "unit": "spline-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": DTYPE[precision], "data": "synthetic",
            "config": workload_config(cfg, world, "gpu", {"precision": PRECISION_NOTE[precision], "steps_per_launch": chunk}),
            "clocks": clocks,
            "e2e": {"value": spline_steps / (ms_e2e * 1e-3), "unit": "spline-steps/s",
                    "h2d_bytes_per_step": h2d * e2e_launches / args.steps,
                    "d2h_bytes_per_step": d2h / args.steps,
                    "includes": "H2D of a/b/omega per launch, the launch, status read-back"
                                + (", NCCL gather of omega+energy on rank 0" if world > 1 else "") + ", D2H of omega+energy"},
            "gpu_launches": launches,
            "roofline": roof,
            "other_modes": other,
        }
        if world == 1 and not args.no_cpu:
            rate, cores, kind, sample = cpu_reference_rate(cfg, steps=2, warmup=1, budget_s=20.0)
            line["cpu_baseline"] = {"value": rate, "unit": "spline-steps/s", "cores": cores, "kind": kind, "sample": sample}
            try:   # the reference's own GPU path (src/optimize.py:81 picks cuda when present): eager fp32 on this B200
                torch.cuda.empty_cache()
                grate, gkind, gsample = reference_loop_rate(cfg, dev, steps=3, warmup=2, sample=min(200, N))
                line["gpu_eager_baseline"] = {"value": grate, "unit": "spline-steps/s", "kind": gkind, "sample": gsample}
            except Exception as exc:  # noqa: BLE001
                line["gpu_eager_baseline"] = {"unavailable": str(exc)[:200]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="vlg", choices=["vlg", "reference"])
    ap.add_argument("--precision", default=None, choices=["f16", "f16x3", "f16x3f", "tf32", "fp32"],
                    help="default: vlg_b200.DEFAULT_PRECISION (the one default of the package and the CLIs)")
    ap.add_argument("--config", type=int, default=3, choices=[2, 3, 5], help="BASELINE.json configuration")
    ap.add_argument("--chunk", type=int, default=50, help="Adam steps per kernel launch")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / gpu_eager_baseline legs")
    ap.add_argument("--no-other", action="store_true", help="skip the secondary arithmetic modes")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed steps computed in their last step (energy, omega, adam_m, adam_v of "
                         "every curve) as DIR/<name>.npy; the inputs are seeded, so two builds compare output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "vlg":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl vlg)")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
