#!/usr/bin/env python
"""Generates tests/golden/flow_small.npz and imu_small.npz from the UNMODIFIED reference (oracle/_ref/libref_mtrack.so, built by
oracle/build_ref.py from /root/reference).  Run in the build container only (needs /root/reference):

    python tests/golden/make_golden.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from flow import SMALL, run_flow, run_imu_rows, save_golden, small_frames  # noqa: E402
from oracle import build_ref, refapi  # noqa: E402

if __name__ == "__main__":
    assert build_ref.build(level_b=False), "reference sources not available"
    f0, f1 = small_frames()
    out = run_flow(refapi.RefMap, SMALL, f0, f1, refapi.so3_exp)
    save_golden(os.path.join(HERE, "flow_small.npz"), dict(f0=f0, f1=f1, **out))
    print("wrote flow_small.npz:", {k: (v.shape, str(v.dtype)[:12]) for k, v in list(out.items())[:6]}, "...")
    print("kn:", out["f0_kn_tresh"], out["f1_kn_tresh"], "dm:", out["dm_count"], "min V:", out["min_V"])
    imu = run_imu_rows(refapi.RefMap, refapi, SMALL, f0, f1)
    np.savez_compressed(os.path.join(HERE, "imu_small.npz"), **imu)
    print("wrote imu_small.npz: TryVel scores", [float(imu["tv%d_score" % i][0]) for i in range(4)], "Minimizer_V",
          imu["mv_V"], "forward matches", imu["er_nfwd"], "ExtRotVel X", imu["er_X"])
