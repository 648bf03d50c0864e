"""CPU suite: pins the oracle.  (1) The CPU restatement oracle/rebvo_oracle.cpp against the golden vectors that
tests/golden/make_golden.py generated from the unmodified reference; (2) the compiled reference itself against
the same vectors when oracle/_ref is present; (3) restatement vs compiled reference on a second, larger seeded
input.  Integer / float32 / per-keyline float64 results are compared bit for bit; only what passes through the
6x6 SVD solve (LAPACK in the reference) gets a 1e-9 tolerance."""
import os

import numpy as np
import pytest

import ctypes as C

from flow import DOG_THRESH, PLANE_FIT, POS_NEG, SMALL, compare, load_golden, run_flow, run_imu_rows, small_frames

GOLD = os.path.join(os.path.dirname(__file__), "golden", "flow_small.npz")
TOL = ("min_V", "min_W", "min_RVel", "min_RW0", "min_W_X", "min_scalars")


@pytest.fixture(scope="module")
def golden():
    return load_golden(GOLD)


def _override(g):
    return dict(V=g["min_V"], W=g["min_W"], RVel=g["min_RVel"], RW0=g["min_RW0"])


def test_golden_inputs_reproducible(golden):
    f0, f1 = small_frames()
    assert np.array_equal(f0, golden["f0"]) and np.array_equal(f1, golden["f1"])


def test_port_matches_golden(golden):
    from oracle import portapi
    out = run_flow(portapi.PortMap, SMALL, golden["f0"], golden["f1"], portapi.so3_exp, _override(golden))
    ref = {k: v for k, v in golden.items() if k not in ("f0", "f1")}
    fails = compare(ref, out, tol_keys=TOL)
    assert not fails, "\n".join(fails)
    # the minimiser itself: same LM path, different 6x6 solver
    assert np.allclose(out["min_V"], golden["min_V"], rtol=1e-9, atol=1e-12)
    assert np.allclose(out["min_W"], golden["min_W"], rtol=1e-9, atol=1e-12)


def test_reference_matches_golden(golden):
    from oracle import refapi
    if not refapi.available():
        pytest.skip("oracle/_ref not built")
    out = run_flow(refapi.RefMap, SMALL, golden["f0"], golden["f1"], refapi.so3_exp, _override(golden))
    ref = {k: v for k, v in golden.items() if k not in ("f0", "f1")}
    fails = compare(ref, out, tol_keys=TOL)
    assert not fails, "\n".join(fails)


def test_port_matches_reference_qvga():
    from oracle import portapi, refapi
    from rebvo_b200 import synth
    if not refapi.available():
        pytest.skip("oracle/_ref not built")
    cfg = dict(SMALL, cam=dict(w=320, h=240, zfx=260.0, zfy=258.0, ppx=161.0, ppy=118.5), kl_max=9000, kl_ref=5000,
               track_points=4000, radius=20, sigma0=3.56359)
    f0, f1 = synth.frame_pair(seed=23, w=320, h=240, nrect=90, shift=(-1.6, 0.9))
    a = run_flow(refapi.RefMap, cfg, f0, f1, refapi.so3_exp)
    ov = dict(V=a["min_V"], W=a["min_W"], RVel=a["min_RVel"], RW0=a["min_RW0"])
    b = run_flow(portapi.PortMap, cfg, f0, f1, portapi.so3_exp, ov)
    fails = compare(a, b, tol_keys=TOL)
    assert not fails, "\n".join(fails)
    assert a["f0_kl"].shape[0] > 2000


def test_kl_max_truncation_and_empty_image():
    """Edge cases of build_mask: the kl_max cut clears the rest of the mask; a flat image yields no keylines."""
    from oracle import portapi
    cam = SMALL["cam"]
    f0, _ = small_frames()
    m = portapi.PortMap(cam["w"], cam["h"], cam["ppx"], cam["ppy"], cam["zfx"], cam["zfy"], 1.7818, 1.2599)
    m.rgb2bw(f0)
    m.build()
    kn_full, _, _ = m.detect(2, 0.4, 0.0952598689, 3000, 0.012, 0, 1500, 0.0, 1, 0)
    full_mask = m.mask().copy()
    kn, _, _ = m.detect(2, 0.4, 0.0952598689, 500, 0.012, 0, 1500, 0.0, 1, 0)
    assert kn == 500 and kn_full > 500
    mask = m.mask()
    assert mask.max() == 499 and (mask >= 0).sum() == 500
    assert np.array_equal(mask[(full_mask >= 0) & (full_mask < 500)], full_mask[(full_mask >= 0) & (full_mask < 500)])
    flat = np.full((cam["h"], cam["w"], 3), 90, np.uint8)
    m.rgb2bw(flat)
    m.build()
    kn, _, _ = m.detect(2, 0.4, 0.0952598689, 3000, 0.012, 0, 1500, 0.0, 1, 0)
    assert kn == 0 and (m.mask() == -1).all()
    assert np.abs(m.plane("dog")).max() < 1e-3


def test_box_plan_known_answers():
    """SURVEY.md 8(a) row D2: Kovesi box widths / achieved sigmas of iigauss::iigauss."""
    from oracle import portapi
    for sigma0, want in ((1.7818, ([3, 3, 5], [3, 5, 5], 1.825742, 2.160247)),
                         (3.56359, ([7, 7, 7], [9, 9, 9], 3.464102, 4.472136))):
        m = portapi.PortMap(64, 64, 32, 32, 50, 50, sigma0, 1.2599)
        d, s = m.box_plan()
        assert d[0].tolist() == want[0] and d[1].tolist() == want[1]
        assert abs(s[0] - want[2]) < 1e-6 and abs(s[1] - want[3]) < 1e-6


def test_port_imu_rows_match_reference():
    """SURVEY.md 8(a) rows K6 / K13 (IMU mode): TryVel, Minimizer_V<double>, ExtRotVel, BiasCorrect restated in the port
    against the unmodified reference on a seeded frame pair.  TryVel is sequential double arithmetic in the reference's
    order: bit-identical, including the in-place residual buffer and the forward-match ids."""
    from oracle import portapi, refapi
    from rebvo_b200 import synth
    if not refapi.available():
        pytest.skip("oracle/_ref not built")
    cam = dict(w=320, h=240, zfx=260.0, zfy=258.0, ppx=161.0, ppy=118.5)
    cfg = dict(SMALL, cam=cam, kl_max=9000, kl_ref=5000, track_points=4000, radius=20, sigma0=3.56359)
    f0, f1 = synth.frame_pair(seed=31, w=320, h=240, nrect=90, shift=(0.5, -0.3))
    mk = lambda cls: [cls(cam["w"], cam["h"], cam["ppx"], cam["ppy"], cam["zfx"], cam["zfy"], cfg["sigma0"],
                          cfg["ksigma"]) for _ in range(2)]
    refs, ports = mk(refapi.RefMap), mk(portapi.PortMap)
    t, l = 0.012, 0
    for r, fr in zip(refs, (f0, f1)):
        r.rgb2bw(fr)
        r.build()
        _, t, l = r.detect(PLANE_FIT, POS_NEG, DOG_THRESH, cfg["kl_max"], t, l, cfg["kl_ref"], cfg["gain"], cfg["tmax"],
                           cfg["tmin"])
    old_r, new_r = refs
    _, rt_new = new_r.reestimate(cfg["track_points"], 100)
    _, rt_old = old_r.reestimate(cfg["track_points"], 100)
    rng = np.random.default_rng(5)
    kl = old_r.keylines()
    assert len(kl) > 1500
    kl["rho"] = rng.uniform(0.7, 1.5, len(kl))
    kl["s_rho"] = rng.uniform(0.05, 0.5, len(kl))
    kl["m_num"] = rng.integers(0, 6, len(kl))
    old_r.set_keylines(kl)
    old_p, new_p = ports
    for pm, rm in ((old_p, old_r), (new_p, new_r)):
        pm.set_keylines(rm.keylines())
        pm.set_mask(rm.mask())
    new_r.build_field(cfg["radius"], rt_new)
    new_p.build_field(cfg["radius"], rt_new)
    q = old_r.quantile(1e-3, 20.0, 0.9, 100)
    res = np.zeros(old_r.knum())
    for V in (np.zeros(3), np.array([0.003, -0.002, 0.004]), np.array([-0.005, 0.001, -0.6])):
        s_r, J_r, F_r, res_r = new_r.try_vel(old_r, V, cfg["match_thresh"], q, 0, res, 2.0, rt_old)
        s_p, J_p, F_p, res_p = new_p.try_vel(old_p, V, cfg["match_thresh"], q, 0, res, 2.0, rt_old)
        assert s_r == s_p and np.array_equal(J_r, J_p) and np.array_equal(F_r, F_p)
        assert np.array_equal(res_r, res_p)
        assert np.array_equal(old_r.keylines()["m_id_f"], old_p.keylines()["m_id_f"])
        assert (old_r.keylines()["m_id_f"] >= 0).sum() > 50
        res = res_r
    m_r = new_r.minimizer_v(old_r, np.zeros(3), cfg["match_thresh"], 5, q, 0, 2.0, rt_old)
    m_p = new_p.minimizer_v(old_p, np.zeros(3), cfg["match_thresh"], 5, q, 0, 2.0, rt_old)
    assert np.allclose(m_r["V"], m_p["V"], rtol=1e-12, atol=1e-15) and np.isclose(m_r["F"], m_p["F"], rtol=1e-12)
    assert np.allclose(m_r["RVel"], m_p["RVel"], rtol=1e-10)
    assert np.array_equal(old_r.keylines()["m_id_f"], old_p.keylines()["m_id_f"])
    # ExtRotVel on the forward matches (the port's elimination solve stands in for SVD<>)
    assert old_r.forward_match(new_r) == old_p.forward_match(new_p) > 50
    ok_r, Wx_r, Rx_r, X_r = new_r.ext_rot_vel(m_r["V"], 1.0, 2.0)
    ok_p, Wx_p, Rx_p, X_p = new_p.ext_rot_vel(m_r["V"], 1.0, 2.0)
    assert ok_r and ok_p
    assert np.allclose(Wx_r, Wx_p, rtol=1e-12, atol=1e-12 * np.abs(Wx_r).max())
    assert np.allclose(X_r, X_p, rtol=1e-7, atol=1e-9 * np.abs(X_r).max())
    assert np.allclose(Rx_r, Rx_p, rtol=1e-7, atol=1e-9 * np.abs(Rx_r).max())
    # BiasCorrect
    R = refapi.lib()
    _p = lambda a: a.ctypes.data_as(C.c_void_p)
    for _ in range(5):
        J = rng.normal(size=(30, 6))
        Wx = J.T @ J + np.eye(6)
        X = rng.normal(size=6) * 1e-2
        Gb = rng.normal(size=3) * 1e-3
        A = rng.normal(size=(3, 3))
        Wb = A @ A.T + np.eye(3) * 10
        Rg = np.ascontiguousarray(np.eye(3) * 1e-4 + 1e-6 * (A @ A.T))
        Rb = np.ascontiguousarray(np.eye(3) * 1e-8)
        b = [np.ascontiguousarray(v.copy()) for v in (X, Wx, Gb, Wb)]
        R.ref_bias_correct(_p(b[0]), _p(b[1]), _p(b[2]), _p(b[3]), _p(Rg), _p(Rb))
        a = portapi.bias_correct(X, Wx, Gb, Wb, Rg, Rb)
        for x, y in zip(a, b):
            assert np.allclose(x, y, rtol=1e-11, atol=1e-14 * max(1.0, np.abs(y).max()))


def test_port_undistort_matches_reference():
    """SURVEY.md 8(f) rank 1: image_undistort map + integer bilinear interpolation, bit for bit, with EuRoC-like and
    exaggerated distortion coefficients (taps that leave the image drop out of the weights)."""
    from oracle import portapi, refapi
    if not refapi.available():
        pytest.skip("oracle/_ref not built")
    cam = dict(w=320, h=240, zfx=260.0, zfy=258.0, ppx=161.0, ppy=118.5)
    rng = np.random.default_rng(9)
    img = rng.integers(0, 256, (cam["h"], cam["w"], 3), dtype=np.uint8)
    for kc in ([-0.28340811, 0.07395907, 0.0, 0.00019359, 1.76187114e-05], [-0.6, 0.3, -0.05, 0.01, -0.02],
               [0.0, 0.0, 0.0, 0.0, 0.0]):
        a = refapi.undistort_rgb(cam, kc, img)
        b = portapi.undistort_rgb(cam, kc, img)
        assert np.array_equal(a, b), "differs in %d bytes" % int((a != b).sum())
    assert not np.array_equal(refapi.undistort_rgb(cam, [-0.6, 0.3, -0.05, 0.01, -0.02], img), img)


GOLD_IMU = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "imu_small.npz")
# bit-exact unless listed: the port's 3x3 / 6x6 solves are restatements of TooN's (1e-12) or stand-ins for SVD<> (1e-7)
IMU_TOL = {"mv_V": 1e-11, "mv_RVel": 1e-9, "mv_F": 1e-11, "er_Rx": 1e-7, "er_X": 1e-7, "er_Wx": 1e-12, "bc_X": 1e-11,
           "bc_Wx": 1e-11, "bc_Gb": 1e-11, "bc_Wb": 1e-11}


def _check_imu(out, gold, tol=None):
    tol = IMU_TOL if tol is None else tol
    fails = []
    for k in gold:
        a, b = gold[k], out[k]
        if k in tol:
            if not np.allclose(a, b, rtol=tol[k], atol=tol[k] * max(1e-300, float(np.abs(a).max()))):
                fails.append("%s: max abs diff %.3e" % (k, float(np.abs(a - b).max())))
        else:   # keyline records: the fields the reference initialises (flow.compare); everything else bit for bit
            fails += compare({k: a}, {k: b})
    return fails


def test_port_imu_rows_match_golden():
    """The IMU-mode rows and the undistortion of the port against vectors generated from the unmodified reference
    (tests/golden/make_golden.py): runs everywhere, with or without oracle/_ref."""
    from oracle import portapi
    z = np.load(GOLD_IMU)
    gold = {k: z[k] for k in z.files}
    f0, f1 = small_frames()
    kls = (gold["imu_old_kl"], gold["imu_new_kl"], gold["imu_old_mask"], gold["imu_new_mask"], gold["imu_retuned"])
    out = run_imu_rows(portapi.PortMap, portapi, SMALL, f0, f1, keylines=kls)
    fails = _check_imu(out, gold)
    assert not fails, "\n".join(fails)
    assert int(gold["er_nfwd"][0]) > 500 and int(gold["er_ok"][0]) == 1


def test_reference_imu_rows_match_golden():
    from oracle import refapi
    if not refapi.available():
        pytest.skip("oracle/_ref not built")
    z = np.load(GOLD_IMU)
    gold = {k: z[k] for k in z.files}
    f0, f1 = small_frames()
    out = run_imu_rows(refapi.RefMap, refapi, SMALL, f0, f1)
    fails = _check_imu(out, gold, tol={})
    assert not fails, "\n".join(fails)
