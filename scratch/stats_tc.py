import sys, os, ctypes
os.environ["VLG_B200_LIB"] = sys.argv[1]
sys.path.insert(0, ".")
import numpy as np, torch
import vlg_b200, bench
from vlg_b200 import _lib
nc = 148
w, a, b, om, _ = bench.synthetic_workload(nc)
dev = "cuda"
dec = vlg_b200.DecoderEnsemble.from_arrays(*[w[k] for k in ("W1", "b1", "W2", "b2", "W3", "b3")], dev)
basis, _ = vlg_b200.construct_nullspace_basis(4)
m = vlg_b200.GeodesicSplineBatch(a.to(dev), b.to(dev), basis.to(dev), om.to(dev), 4)
t = torch.linspace(0, 1, 2000, device=dev)
for _ in range(2):
    vlg_b200.optimize_splines(m, dec, t, 1, M=2, seed=0, precision=(sys.argv[2] if len(sys.argv) > 2 else "tf32"))
torch.cuda.synchronize()
lib = _lib.load()
out = (ctypes.c_longlong * (nc * 8))()
lib.vlg_debug_tc_stats.argtypes = [ctypes.c_void_p, ctypes.c_int]
assert lib.vlg_debug_tc_stats(out, nc) == 0
st = np.array(out).reshape(nc, 8).astype(np.float64)
names = ["setup warp busy", "setup warp wait buffer", "mma wait full", "mma total", "epi0 wait acc", "mma issue loops", "epi1 wait acc", "-"]
for i, nm in enumerate(names):
    if nm != "-":
        print(f"{nm:22s} mean {st[:, i].mean():12.0f} cycles  ({100 * st[:, i].mean() / st[:, 3].mean():5.1f}% of mma total)")


if not hasattr(lib, "vlg_debug_tc_phase"):
    sys.exit(0)
ph = (ctypes.c_longlong * (nc * 48))()
lib.vlg_debug_tc_phase.argtypes = [ctypes.c_void_p, ctypes.c_int]
assert lib.vlg_debug_tc_phase(ph, nc) == 0
ph = np.array(ph).reshape(nc, 2, 24).astype(np.float64).mean(0)
names = ["F: item setup + sw wait", "F: layer 1 + st + arrive", "F: wait F2", "F: E-F2", "F: wait F3", "F: E-F3",
         "window setup (points, wait lists)", "bar after forward", "energy pass", "B: setup + G build + arrive", "B: wait B3", "B: E-B3",
         "B: wait B2", "B: E-B2 (dz)", "bar after backward", "domega + reductions", "step prologue/Adam", "-", "-", "-", "e: loads + diff loop", "e: warp sum", "d: first barrier", "d: design rows + warp sums + bar"]
for c in range(2):
    tot = ph[c].sum()
    print(f"chain {c}: total {tot:.0f} cycles")
    for i, nm in enumerate(names):
        if nm != "-":
            print(f"   {nm:28s} {ph[c, i]:10.0f}  {100 * ph[c, i] / tot:5.1f}%")
