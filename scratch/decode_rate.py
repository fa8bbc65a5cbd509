"""Rate of the decoder-ensemble op (DecoderEnsemble.__call__ and its backward) against eager PyTorch fp32.

P = 2^20 points uniform in the latent box [-3.5, 3.5]^2, the committed eVAE seed-12 decoders (K = 10, X = 50).
Timed paths: forward, and forward + backward (dz for dx = 1), in f16x3, f16x3f, f16 and fp32, and the same two in eager
PyTorch fp32 (torch.stack of nn.Linear MLPs, autograd to z; TF32 matmuls off, torch's default).  CUDA events, median
of --runs runs per path, the paths alternated.  The output alone (K P X fp32 = 2.1 GB) is larger than L2, so each
run reads its weights and z from L2 or HBM as a user's call would.  Reports point-decoders/s, the FLOP/s of the
shape-computed operation count, the bytes the op must write, and which of compute (the data sheet's dense fp16 tensor
rate; tensor-core paths) or output bandwidth bounds the run.  Prints the card name and power limit of the same run.

    python scratch/decode_rate.py [--runs 7]
"""
import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import vlg_b200  # noqa: E402
from tests import helpers as Hh  # noqa: E402

HBM_BPS = 7.7e12


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=7)
    ap.add_argument("--points", type=int, default=1 << 20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a B200"
    dev = "cuda"
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()[0]
    arrs = Hh.decoder_arrays(Hh.load("evae_seed12_decoders"))
    K, X, P = arrs["W1"].shape[0], arrs["W3"].shape[1], args.points
    ens = vlg_b200.DecoderEnsemble.from_arrays(*[arrs[k] for k in Hh.DEC_KEYS], dev)
    z = (torch.rand((P, 2), device=dev, generator=torch.Generator(dev).manual_seed(0)) * 7.0 - 3.5)

    nets = []
    for k in range(K):
        net = torch.nn.Sequential(torch.nn.Linear(2, 128), torch.nn.ReLU(), torch.nn.Linear(128, 128), torch.nn.ReLU(),
                                  torch.nn.Linear(128, X)).to(dev)
        with torch.no_grad():
            for li, (w, b) in zip((0, 2, 4), (("W1", "b1"), ("W2", "b2"), ("W3", "b3"))):
                net[li].weight.copy_(torch.tensor(arrs[w][k]))
                net[li].bias.copy_(torch.tensor(arrs[b][k]))
        nets.append(net.requires_grad_(False))
    torch.backends.cuda.matmul.allow_tf32 = False

    def vlg_fwd(prec):
        return lambda: ens(z, precision=prec, check=False)

    def vlg_fb(prec):
        def run():
            zz = z.detach().requires_grad_(True)
            ens(zz, precision=prec, check=False).sum().backward()
        return run

    def eager_fwd():
        with torch.no_grad():
            return torch.stack([n(z) for n in nets])

    def eager_fb():
        zz = z.detach().requires_grad_(True)
        torch.stack([n(zz) for n in nets]).sum().backward()

    paths = {f"{p} fwd": vlg_fwd(p) for p in ("f16x3", "f16x3f", "f16", "fp32")}
    paths.update({f"{p} fwd+bwd": vlg_fb(p) for p in ("f16x3", "f16x3f", "f16", "fp32")})
    paths.update({"eager fp32 fwd": eager_fwd, "eager fp32 fwd+bwd": eager_fb})
    times = {k: [] for k in paths}
    for f in paths.values():   # warm-up: module loads, cuBLAS algorithm choice
        f()
    torch.cuda.synchronize()
    for _ in range(args.runs):
        for k, f in paths.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) * 1e-3)

    flop_fwd = 2 * (2 * 128 + 128 * 128 + 128 * X) * P * K                 # per point-decoder: three layers
    flop_bwd = flop_fwd + 2 * (X * 128 + 128 * 128 + 128 * 2) * P * K      # recomputed forward + input gradient
    out_bytes = 4 * K * P * X
    res = {"card": card, "P": P, "K": K, "X": X, "runs": args.runs}
    for k, ts in times.items():
        t = statistics.median(ts)
        bwd = "bwd" in k
        flop = flop_bwd if bwd else flop_fwd
        wbytes = out_bytes                                     # fwd: x written; fwd+bwd: x written, dx read
        rbytes = out_bytes if bwd else 0
        t_bw = (wbytes + rbytes) / HBM_BPS
        r = {"ms": round(t * 1e3, 3), "point_decoders_per_s": K * P / t, "TFLOP_s": flop / t / 1e12,
             "GB_written": wbytes / 1e9, "bandwidth_share": t_bw / t}
        if not (k.startswith("fp32") or k.startswith("eager")):   # fp16 dense tensor rate of the data sheet
            t_comp = flop / 2.25e15
            r.update(bound="compute" if t_comp > t_bw else "output bandwidth", share_of_bound=max(t_comp, t_bw) / t)
        res[k] = r
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
