"""Leaf kernel timing (development aid): batched 128x128 Cholesky+inverse through gpe_potrf with the
per-category CUDA-event profile."""
import os, sys
import numpy as np
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from gp_emu_uqsa_b200 import _lib
B = int(sys.argv[1]) if len(sys.argv) > 1 else 32
rng = np.random.default_rng(0)
M = rng.normal(size=(B, 128, 128)); A = M @ M.transpose(0, 2, 1) + 128 * np.eye(128)
dev = _lib.Device(0)
dev.dbg_potrf_inv(A)
dev.profile_enable(True); dev.profile_read(reset=True)
for _ in range(5):
    Li, ld, st = dev.dbg_potrf_inv(A)
pr = dev.profile_read()
ms, cnt = pr["potrf_leaf"]
err = np.abs(Li[0] @ np.linalg.cholesky(A[0]) - np.eye(128)).max()
print("leaf %.1f us per launch (%d launches), |Linv L - I| = %.2e" % (ms / cnt * 1e3, cnt, err))
