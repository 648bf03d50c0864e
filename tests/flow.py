"""One deterministic two-frame pass through every stage of the edge pipeline, written against the common
interface of oracle.refapi.RefMap (unmodified reference) and oracle.portapi.PortMap (CPU restatement).
Used to generate the golden vectors (tests/golden/make_golden.py) and to check the oracles against them."""
import numpy as np

SMALL = dict(cam=dict(w=160, h=120, zfx=120.0, zfy=118.0, ppx=80.5, ppy=59.25), sigma0=1.7818, ksigma=1.2599,
             thresh=0.012, gain=1e-6, tmax=0.05, tmin=0.005, kl_max=3000, kl_ref=1500, track_points=1200,
             radius=12, match_thresh=0.5, iter_max=4, init_type=2, init_iter=2, reweight=2.0, match_num_thresh=0,
             thr_mod=1.0, thr_ang=45.0, loc_unc_match=2.0, reg_thresh=0.5, q_abs=1e-4, loc_unc=1.0)
POS_NEG, DOG_THRESH, PLANE_FIT = 0.4, 0.095259868922420, 2


def small_frames(cfg=SMALL, seed=11):
    from rebvo_b200 import synth
    cam = cfg["cam"]
    return synth.frame_pair(seed=seed, w=cam["w"], h=cam["h"], nrect=40, shift=(1.25, -0.6))


def seed_depth(kl, seed=5):
    rng = np.random.default_rng(seed)
    kl = kl.copy()
    kl["rho"] = rng.uniform(0.6, 1.6, len(kl))
    kl["s_rho"] = rng.uniform(0.05, 0.6, len(kl))
    kl["m_num"] = rng.integers(0, 7, len(kl))
    return kl


def run_flow(Map, cfg, f0, f1, so3_exp, minim_override=None):
    """Returns {name: array}.  minim_override: dict(V, W, RVel) to feed the post-minimiser stages with fixed
    inputs (so that everything downstream is comparable bit for bit even if the 6x6 solver differs)."""
    cam = cfg["cam"]
    maps = [Map(cam["w"], cam["h"], cam["ppx"], cam["ppy"], cam["zfx"], cam["zfy"], cfg["sigma0"], cfg["ksigma"])
            for _ in range(2)]
    out = {}
    t, l = cfg["thresh"], 0
    for i, fr in enumerate((f0, f1)):
        m = maps[i]
        m.rgb2bw(fr)
        m.build()
        for pl in ("gray", "img0", "img1", "dog"):
            out["f%d_%s" % (i, pl)] = m.plane(pl)
        out["f%d_dx" % i] = m.plane("dx")[1:-1, 1:-1].copy()
        out["f%d_dy" % i] = m.plane("dy")[1:-1, 1:-1].copy()
        kn, t, l = m.detect(PLANE_FIT, POS_NEG, DOG_THRESH, cfg["kl_max"], t, l, cfg["kl_ref"], cfg["gain"],
                            cfg["tmax"], cfg["tmin"])
        out["f%d_kn_tresh" % i] = np.array([kn, t, l], np.float64)
        out["f%d_kl" % i] = m.keylines()
        out["f%d_mask" % i] = m.mask()
        out["f%d_retuned" % i] = np.array([m.reestimate(cfg["track_points"], 100)[1]], np.float32)
    old, new = maps
    old.set_keylines(seed_depth(old.keylines()))
    q = old.quantile(1e-3, 20.0, 0.9, 100)
    out["quantile"] = np.array([q])
    new.build_field(cfg["radius"], float(out["f1_retuned"][0]))
    fld = new.field()
    out["field_ikl"] = fld[:, :, 1].copy()
    out["field_dist"] = np.where(fld[:, :, 1] >= 0, fld[:, :, 0], -1)
    k0 = old.knum()
    pnum = (k0 + 3) & ~3
    res_prev = np.zeros(pnum)
    Xs = [np.zeros(6), np.array([0.004, -0.002, 0.001, 0.002, -0.003, 0.004])]
    for xi, X in enumerate(Xs):
        for (rw, pj) in ((False, True), (True, True), (True, False)):
            s, J, F, res = new.try_vel_rot(old, X, rw, pj, cfg["match_thresh"], q, cfg["match_num_thresh"],
                                           cfg["reweight"], res_prev)
            tag = "tvr_x%d_rw%d_pj%d" % (xi, rw, pj)
            out[tag + "_score"] = np.array([s])
            if pj:
                out[tag + "_JtJ"], out[tag + "_JtF"] = J, F
            kl_old = old.keylines()
            out[tag + "_m_id_f"] = kl_old["m_id_f"].copy()
            used = kl_old["s_rho"] <= q
            out[tag + "_res"] = np.where(used, res[:k0], 0.0)
            if pj and not rw:
                res_prev = np.where(np.isfinite(res), res, 0.0)
    mr = new.minimizer_rv(old, np.zeros(3), np.zeros(3), cfg["match_thresh"], cfg["iter_max"], cfg["init_type"],
                          cfg["reweight"], q, cfg["match_num_thresh"], cfg["init_iter"])
    for k in ("V", "W", "RVel", "RW0", "W_X"):
        out["min_" + k] = np.array(mr[k])
    out["min_scalars"] = np.array([mr["F"], mr["rel_err"], mr["rel_err_score"]])
    out["min_m_id_f"] = old.keylines()["m_id_f"].copy()
    if minim_override is not None:
        mr = dict(mr, **minim_override)
    old.forward_match(new)
    out["fm_kl"] = new.keylines()
    R0 = so3_exp(mr["W"])
    old.rotate(R0)
    out["rot_kl"] = old.keylines()
    n = new.directed_matching(old, mr["V"], mr["RVel"], R0.T.copy(), cfg["thr_mod"], cfg["thr_ang"], cfg["radius"],
                              cfg["loc_unc_match"])
    out["dm_count"] = np.array([n])
    out["dm_kl"] = new.keylines()
    out["reg_count"] = np.array([new.regularize(cfg["reg_thresh"])])
    out["reg_kl"] = new.keylines()
    new.ekf(mr["V"], mr["RVel"], mr["RW0"], cfg["q_abs"], 1.6968e-4, cfg["loc_unc"])
    out["ekf_kl"] = new.keylines()
    out["rescale"] = np.array(new.rescale(20.0, 1, False))
    return out


# fields of KeyLine that the reference defines (m_m0/n_m0/score are stack garbage until a match is copied)
KL_FIELDS = ["p_inx", "m_m", "u_m", "n_m", "c_p", "rho", "s_rho", "rho_nr", "s_rho_nr", "rho0", "s_rho0", "p_m",
             "p_m_0", "m_id", "m_id_f", "m_id_kf", "m_num", "p_id", "n_id"]


# keyline arrays of the later stages and the array each one was derived from (parents first)
KL_PARENT = {"rot_kl": "f0_kl", "fm_kl": "f1_kl", "dm_kl": "fm_kl", "reg_kl": "dm_kl", "ekf_kl": "reg_kl"}


def save_golden(path, arrays):
    """np.savez layout with LZMA members (np.load reads it).  A keyline array of KL_PARENT is stored as only the fields
    that differ from its parent's, under "<name>.<field>": together this keeps the file under 1 MB."""
    import io
    import zipfile
    with zipfile.ZipFile(path, "w", zipfile.ZIP_LZMA) as zf:
        def put(name, a):
            buf = io.BytesIO()
            np.save(buf, np.ascontiguousarray(a))
            zf.writestr(name + ".npy", buf.getvalue())
        for k, a in arrays.items():
            if k not in KL_PARENT:
                put(k, a)
                continue
            parent = arrays[KL_PARENT[k]]
            assert len(parent) == len(a), k
            for f in a.dtype.names:
                if a[f].tobytes() != parent[f].tobytes():
                    put("%s.%s" % (k, f), a[f])


def load_golden(path):
    """The arrays save_golden wrote, keyline arrays of KL_PARENT rebuilt whole."""
    z = np.load(path)
    out = {k: z[k] for k in z.files if "." not in k}
    for k, parent in KL_PARENT.items():
        a = out[parent].copy()
        for f in a.dtype.names:
            if "%s.%s" % (k, f) in z.files:
                a[f] = z["%s.%s" % (k, f)]
        out[k] = a
    return out


def compare(ref, got, tol_keys=(), rtol=1e-9, loose=()):
    """Bitwise comparison of two flow outputs except for keys starting with a prefix in tol_keys.  Returns a list
    of failure strings."""
    fails = []
    for k, a in ref.items():
        b = got[k]
        if a.dtype.names:
            if len(a) != len(b):
                fails.append("%s: kn %d vs %d" % (k, len(a), len(b)))
                continue
            matched = a["m_id"] >= 0
            for f in KL_FIELDS + ["m_m0", "n_m0"]:
                x, y = a[f], b[f]
                if f in ("m_m0", "n_m0"):
                    x, y = x[matched], y[matched]
                if x.dtype.kind == "f" and any(k.startswith(p) for p in loose):
                    ok = np.allclose(x, y, rtol=rtol, atol=1e-12, equal_nan=True)
                else:
                    ok = np.array_equal(x, y, equal_nan=x.dtype.kind == "f")
                if not ok:
                    fails.append("%s.%s differs (%d elements)" % (k, f, int((x != y).sum())))
        elif any(k.startswith(p) for p in tol_keys):
            if not np.allclose(a, b, rtol=rtol, atol=rtol * max(1e-300, float(np.abs(a).max()))):
                fails.append("%s: max abs diff %.3e" % (k, float(np.abs(a - b).max())))
        else:
            same = np.array_equal(a, b, equal_nan=a.dtype.kind == "f")
            if not same:
                fails.append("%s differs in %d elements" % (k, int((a != b).sum())))
    return fails


def run_imu_rows(Map, api, cfg, f0, f1, keylines=None):
    """IMU-mode rows (SURVEY.md 8(a) K6, K13) + undistort (8(f) rank 1) on the same frame pair.  `api` is the module
    that owns Map (oracle.refapi / oracle.portapi): it provides undistort_rgb and bias_correct.  keylines: optional
    (old, new, masks, retuned) taken from the golden file so that a map class without a detector pass can be fed."""
    cam = cfg["cam"]
    old, new = [Map(cam["w"], cam["h"], cam["ppx"], cam["ppy"], cam["zfx"], cam["zfy"], cfg["sigma0"], cfg["ksigma"])
                for _ in range(2)]
    out = {}
    if keylines is None:
        t, l, rt = cfg["thresh"], 0, []
        for m, fr in ((old, f0), (new, f1)):
            m.rgb2bw(fr)
            m.build()
            _, t, l = m.detect(PLANE_FIT, POS_NEG, DOG_THRESH, cfg["kl_max"], t, l, cfg["kl_ref"], cfg["gain"],
                               cfg["tmax"], cfg["tmin"])
            rt.append(m.reestimate(cfg["track_points"], 100)[1])
        old.set_keylines(seed_depth(old.keylines()))
    else:
        k_old, k_new, m_old, m_new, rt = keylines
        old.set_keylines(k_old)
        old.set_mask(m_old)
        new.set_keylines(k_new)
        new.set_mask(m_new)
    out["imu_old_kl"], out["imu_new_kl"] = old.keylines(), new.keylines()
    out["imu_old_mask"], out["imu_new_mask"] = old.mask(), new.mask()
    out["imu_retuned"] = np.array(rt, np.float32)
    new.build_field(cfg["radius"], float(rt[1]))
    q = old.quantile(1e-3, 20.0, 0.9, 100)
    res = np.zeros(old.knum())
    # the last velocity drives 1/rho + Vz negative for the nearer keylines (TryVel's z_p <= 0 branch)
    for vi, V in enumerate((np.zeros(3), np.array([0.004, -0.003, 0.005]), np.array([-0.006, 0.002, -0.55]),
                            np.array([0.001, 0.0, -0.7]))):
        s, J, F, res = new.try_vel(old, V, cfg["match_thresh"], q, 0, res, cfg["reweight"], float(rt[0]))
        out["tv%d_score" % vi], out["tv%d_JtJ" % vi], out["tv%d_JtF" % vi] = np.array([s]), J, F
        out["tv%d_res" % vi], out["tv%d_m_id_f" % vi] = res.copy(), old.keylines()["m_id_f"].copy()
    mv = new.minimizer_v(old, np.zeros(3), cfg["match_thresh"], 5, q, 0, cfg["reweight"], float(rt[0]))
    out["mv_V"], out["mv_RVel"], out["mv_F"] = np.array(mv["V"]), np.array(mv["RVel"]), np.array([mv["F"]])
    out["mv_m_id_f"] = old.keylines()["m_id_f"].copy()
    out["er_nfwd"] = np.array([old.forward_match(new)])
    ok, Wx, Rx, X = new.ext_rot_vel(out["mv_V"], cfg["loc_unc"], cfg["reweight"])
    out["er_ok"], out["er_Wx"], out["er_Rx"], out["er_X"] = np.array([int(ok)]), Wx, Rx, X
    rng = np.random.default_rng(4)
    Jm = rng.normal(size=(30, 6))
    A = rng.normal(size=(3, 3))
    bc = api.bias_correct(rng.normal(size=6) * 1e-2, Jm.T @ Jm + np.eye(6), rng.normal(size=3) * 1e-3,
                          A @ A.T + np.eye(3) * 10, np.eye(3) * 1e-4 + 1e-6 * (A @ A.T), np.eye(3) * 1e-8)
    out["bc_X"], out["bc_Wx"], out["bc_Gb"], out["bc_Wb"] = bc
    out["und"] = api.undistort_rgb(cam, [-0.28340811, 0.07395907, 0.0, 0.00019359, 1.76187114e-05], f0)
    return out

