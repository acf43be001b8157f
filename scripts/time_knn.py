"""Timing of K2 at several k-NN grid cell edges on the bench workload (one process):
    python scripts/time_knn.py [pairs] [cells...]      cell = k-NN grid cell edge in m (gicpParams.knn_cell), 0 = auto
Prints the knn_cov stage time (CUDA events inside the library) and the largest covariance difference
against the first cell edge."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
from generalized_icp_b200 import synthetic  # noqa: E402
from generalized_icp_b200.engine import GicpEngine  # noqa: E402

pairs = int(sys.argv[1]) if len(sys.argv) > 1 else 256
cells = sys.argv[2:] or ["0", "1.0", "1.6"]
cfg = {k: v for k, v in synthetic.CONFIG4.items() if k != "n"}
src, tgt, off, _ = synthetic.patches3d_batch_device(pairs, n=32768, seed=0, device="cuda", **cfg)
off = off.cpu().numpy()
eng = GicpEngine(3, "f32")
ref = None
for cell in cells:
    eng.set_params(**synthetic.CONFIG4_PARAMS, knn_cell=float(cell))
    for _ in range(2):
        eng.set_target(tgt, off)
    eng.profile(True)
    for _ in range(3):
        eng.set_target(tgt, off)
    prof = eng.profile_read()
    eng.profile(False)
    cov = eng.covariances(1)
    if ref is None:
        ref = cov
    diff = float((cov - ref).abs().max())
    nbad = int(((cov - ref).abs().amax(dim=(1, 2)) > 1e-3).sum())
    print(f"cell={cell:>5s}  knn_cov {prof['knn_cov'][0] / 3:8.3f} ms  grid {prof['grid_build'][0] / 3:7.3f} ms"
          f"  max|dC| {diff:.2e}  points off by >1e-3: {nbad}", flush=True)
