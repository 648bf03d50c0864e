"""Drop-in boundary test: tests/shim_driver.cpp = the reference's FirstThr/SecondThread call sequence written
against include/rebvo_b200_shim.hpp (same class and method names as the reference's mtracklib) and compiled with
the reference's non-hot-path headers.  Its trajectory must equal rb_pipeline_push's and the reference's."""
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
NF = 30


def test_shim_classes_reproduce_reference_flow(built, tmp_path):
    from oracle import refapi
    from rebvo_b200 import capi, synth
    exe = os.path.join(os.path.dirname(refapi.EXE), "shim_driver")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/shim_driver not built (needs the reference headers)")
    cam = synth.EUROC
    seq = synth.Sequence(w=cam["w"], h=cam["h"], seed=9, zf=cam["zfx"])
    ts, fr = seq.frames(NF)
    path = str(tmp_path / "frames.bin")
    synth.write_frames_file(path, ts, fr)
    r = subprocess.run([refapi.runnable(exe), path, path + ".shim"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    with open(path + ".shim", "rb") as f:
        n, sz = np.frombuffer(f.read(8), np.int32)
        assert sz == refapi.OUTREC.itemsize
        shim = np.frombuffer(f.read(), refapi.OUTREC, count=n)
    pl = capi.Pipeline(capi.default_params(cam), max_batch=10)
    nav = np.concatenate([pl.push(fr[s:s + 10], ts[s:s + 10]) for s in range(0, NF, 10)])
    pl.close()
    assert len(shim) == NF
    assert np.array_equal(shim["kn"], nav["kn"])
    assert np.array_equal(shim["matches"][1:], nav["matches"][1:])
    d = np.abs(shim["Pos"] - nav["Pos"]).max()
    print("shim vs pipeline max |dPos| %.3e" % d)
    assert d <= 1e-9
    assert np.abs(shim["PoseLie"] - nav["PoseLie"]).max() <= 1e-9
    if os.path.exists(refapi.EXE):
        info, rec = refapi.run_full_rebvo(path, path + ".ref")
        m = min(len(rec), NF - 1)
        assert np.array_equal(rec["kn"][:m], shim["kn"][:m])
        ate = float(np.sqrt(((rec["Pos"][:m] - shim["Pos"][:m]) ** 2).sum(1).mean()))
        print("shim vs reference ATE %.3e m" % ate)
        assert ate <= 1e-7
