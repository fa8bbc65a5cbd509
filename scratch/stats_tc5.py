"""Phase statistics (VLG_TC_STATS build) on the config-5 shape: 148 groups of 7 curves, K=64, T=256, n_poly=8."""
import sys, os, ctypes
os.environ["VLG_B200_LIB"] = sys.argv[1]
sys.path.insert(0, ".")
import numpy as np, torch
import vlg_b200, bench
from vlg_b200 import _lib
prec = sys.argv[2] if len(sys.argv) > 2 else "f16"
nc = 148
N, K, n_poly, T = 148 * 7, 64, 8, 256
w = bench.random_decoders(K, 0)
g = torch.Generator().manual_seed(0)
a = torch.rand(N, 2, generator=g) * 6 - 3; b = torch.rand(N, 2, generator=g) * 6 - 3
om = 0.1 * torch.randn(N, n_poly + 1, 2, generator=g)
dev = "cuda"
dec = vlg_b200.DecoderEnsemble.from_arrays(*[w[k] for k in ("W1", "b1", "W2", "b2", "W3", "b3")], dev)
basis, _ = vlg_b200.construct_nullspace_basis(n_poly)
m = vlg_b200.GeodesicSplineBatch(a.to(dev), b.to(dev), basis.to(dev), om.to(dev), n_poly)
t = torch.linspace(0, 1, T, device=dev)
for _ in range(2):
    vlg_b200.optimize_splines(m, dec, t, 1, M=2, seed=0, precision=prec)
torch.cuda.synchronize()
lib = _lib.load()
ph = (ctypes.c_longlong * (nc * 48))()
lib.vlg_debug_tc_phase.argtypes = [ctypes.c_void_p, ctypes.c_int]
assert lib.vlg_debug_tc_phase(ph, nc) == 0
ph = np.array(ph).reshape(nc, 2, 24).astype(np.float64).mean(0)
names = ["F: item setup + sw wait", "F: layer 1 + st + arrive", "F: wait F2", "F: E-F2", "F: wait F3", "F: E-F3",
         "window setup (points, wait lists)", "bar after forward", "energy pass (+ tile pass)", "B: setup + G build + arrive", "B: wait B3", "B: E-B3",
         "B: wait B2", "B: E-B2 (dz)", "bar after backward", "domega + reductions", "step prologue/Adam",
         "-", "-", "-", "e: loads + diff loop", "e: warp sum", "d: first barrier", "d: design rows + warp sums + bar"]
for c in range(1):
    tot = ph[c].sum()
    print(f"chain {c}: total {tot:.0f} cycles per group-step (7 curves)")
    for i, nm in enumerate(names):
        print(f"   {nm:40s} {ph[c, i]:10.0f}  {100 * ph[c, i] / tot:5.1f}%")
