"""GPU: `bench.py --dump-outputs` writes what its timed steps computed: the same arrays, bit for bit, as the
public API returns for warm-up + timed steps of the same seeded workload."""
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from tests import helpers as Hh

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def test_dumped_outputs_are_the_last_timed_step(tmp_path, built_lib):
    import bench
    import vlg_b200
    warmup, steps = 3, 2
    out = tmp_path / "outputs"
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", str(steps), "--warmup", str(warmup),
                          "--no-cpu", "--no-other", "--dump-outputs", str(out)],
                         cwd=tmp_path, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout + res.stderr
    cfg = bench.make_config(3)
    dev = "cuda"
    dec = vlg_b200.DecoderEnsemble.from_arrays(*[cfg["w"][k] for k in Hh.DEC_KEYS], dev)
    basis = vlg_b200.construct_nullspace_basis(cfg["n_poly"])[0].to(dev)
    model = vlg_b200.GeodesicSplineBatch(cfg["a"].to(dev), cfg["b"].to(dev), basis, cfg["omega"].to(dev), cfg["n_poly"])
    t = torch.linspace(0, 1, cfg["T"], device=dev)
    for _ in range(warmup):
        vlg_b200.optimize_splines(model, dec, t, 1, M=cfg["M"], seed=0)
    energy = vlg_b200.optimize_splines(model, dec, t, steps, M=cfg["M"], seed=0)
    want = {"energy": energy, "omega": model.omega, "adam_m": model.adam_m, "adam_v": model.adam_v}
    assert sorted(p.name for p in out.iterdir()) == sorted(f"{k}.npy" for k in want)
    for name, x in want.items():
        got = np.load(out / f"{name}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, x.cpu().numpy()), name
