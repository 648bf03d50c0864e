"""TEST INFRASTRUCTURE ONLY: ctypes binding of oracle/_ref/libref_mtrack.so (the unmodified reference
mtracklib compiled by oracle/build_ref.py).  Only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / reference arm may import this module; the product never does."""
import atexit
import ctypes as C
import os
import re
import shutil
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "_ref", "libref_mtrack.so")
EXE = os.path.join(HERE, "_ref", "ref_rebvo")

# struct KeyLine, include/mtracklib/edge_finder.h:45-91 (168 bytes, SURVEY.md 8(a) T1)
KEYLINE = np.dtype({
    "names": ["p_inx", "m_m", "u_m", "n_m", "score", "c_p", "rho", "s_rho", "rho_nr", "s_rho_nr",
              "rho0", "s_rho0", "p_m", "p_m_0", "m_id", "m_id_f", "m_id_kf", "m_num", "m_m0", "n_m0",
              "p_id", "n_id", "net_id", "stereo_m_id", "stereo_rho", "stereo_s_rho"],
    "formats": ["i4", ("f4", 2), ("f4", 2), "f4", "f4", ("f4", 2), "f8", "f8", "f8", "f8", "f8", "f8",
                ("f4", 2), ("f4", 2), "i4", "i4", "i4", "i4", ("f4", 2), "f8", "i4", "i4", "i4", "i4",
                "f8", "f8"],
    "offsets": [0, 4, 12, 20, 24, 28, 40, 48, 56, 64, 72, 80, 88, 96, 104, 108, 112, 116, 120, 128,
                136, 140, 144, 148, 152, 160],
    "itemsize": 168})

_lib = None


def _blas_dir():
    import glob
    import importlib.util
    spec = importlib.util.find_spec("cv2")
    return os.path.join(os.path.dirname(os.path.dirname(spec.origin)), "opencv_python_headless.libs")


def _preload():
    import glob
    d = _blas_dir()
    for pat in ("libquadmath*", "libgfortran*", "libopenblas*"):
        for f in sorted(glob.glob(os.path.join(d, pat))):
            C.CDLL(f, mode=C.RTLD_GLOBAL)


def available():
    return os.path.exists(LIB)


def lib():
    global _lib
    if _lib is None:
        _preload()
        _lib = C.CDLL(LIB)
        L = _lib
        L.ref_map_create.restype = C.c_void_p
        L.ref_map_create.argtypes = [C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float,
                                     C.c_double, C.c_double]
        L.ref_quantile.restype = C.c_double
        L.ref_minimizer_rv.restype = C.c_double
        L.ref_try_vel_rot.restype = C.c_double
        L.ref_rescale.restype = C.c_double
        assert L.ref_sizeof_keyline() == KEYLINE.itemsize
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class RefMap:
    """One ring slot of the reference: sspace + edge_tracker + global_tracker (rebvo.cpp:297-312)."""

    def __init__(self, w, h, ppx, ppy, zfx, zfy, sigma0, ksigma):
        self.w, self.h = w, h
        self.L = lib()
        self.h_ = C.c_void_p(self.L.ref_map_create(w, h, ppx, ppy, zfx, zfy, sigma0, ksigma))

    def __del__(self):
        if getattr(self, "h_", None):
            self.L.ref_map_destroy(self.h_)
            self.h_ = None

    def rgb2bw(self, rgb):
        rgb = np.ascontiguousarray(rgb, np.uint8)
        self.L.ref_rgb2bw(self.h_, _p(rgb))

    def set_gray(self, g):
        g = np.ascontiguousarray(g, np.float32)
        self.L.ref_set_gray(self.h_, _p(g))

    def build(self):
        self.L.ref_build(self.h_)

    def plane(self, which):
        idx = {"img0": 0, "img1": 1, "dog": 2, "dx": 3, "dy": 4, "gray": 5}[which]
        out = np.empty((self.h, self.w), np.float32)
        self.L.ref_get_plane(self.h_, idx, _p(out))
        return out

    def detect(self, plane_fit, pos_neg, dog_thresh, kl_max, tresh, l_kl_num, kl_ref, gain, tmax, tmin):
        t = C.c_double(tresh)
        l = C.c_int(l_kl_num)
        kn = self.L.ref_detect(self.h_, plane_fit, C.c_double(pos_neg), C.c_double(dog_thresh), kl_max,
                               C.byref(t), C.byref(l), kl_ref, C.c_double(gain), C.c_double(tmax),
                               C.c_double(tmin))
        return kn, t.value, l.value

    def reestimate(self, knum, n):
        o = C.c_float(0)
        r = self.L.ref_reestimate(self.h_, knum, n, C.byref(o))
        return r, o.value

    def knum(self):
        return self.L.ref_knum(self.h_)

    def keylines(self):
        out = np.zeros(self.knum(), KEYLINE)
        self.L.ref_get_keylines(self.h_, _p(out))
        return out

    def pack_net(self, k_prof=1.0):
        """The reference's wire packer (copy_net_keyline + copy_net_keyline_nextid): uint8 [n, 15]."""
        assert self.L.ref_sizeof_net_keyline() == 15
        out = np.zeros((max(self.knum(), 1), 15), np.uint8)
        n = self.L.ref_pack_net(self.h_, _p(out), len(out), C.c_double(k_prof))
        return out[:n]

    def set_keylines(self, kl):
        kl = np.ascontiguousarray(kl, KEYLINE)
        self.L.ref_set_keylines(self.h_, _p(kl), len(kl))

    def mask(self):
        out = np.empty((self.h, self.w), np.int32)
        self.L.ref_get_mask(self.h_, _p(out))
        return out

    def set_mask(self, mask, kn):
        mask = np.ascontiguousarray(mask, np.int32)
        self.L.ref_set_mask(self.h_, _p(mask), kn)

    def quantile(self, smin, smax, perc, n):
        return self.L.ref_quantile(self.h_, C.c_double(smin), C.c_double(smax), C.c_double(perc), n)

    def build_field(self, radius, min_mod):
        self.L.ref_build_field(self.h_, radius, C.c_float(min_mod))

    def field(self):
        out = np.empty((self.h, self.w, 2), np.int32)
        self.L.ref_get_field(self.h_, _p(out))
        return out

    def minimizer_rv(self, old, V, W, match_thresh, iter_max, init_type, reweight, max_s_rho,
                     match_num_thresh, init_iter):
        V = np.array(V, np.float64)
        W = np.array(W, np.float64)
        RV = np.eye(3) * 1e50
        RW = np.eye(3) * 1e50
        WX = np.zeros((6, 6))
        e1, e2 = C.c_double(0), C.c_double(0)
        F = self.L.ref_minimizer_rv(self.h_, old.h_, _p(V), _p(W), _p(RV), _p(RW), C.c_double(match_thresh),
                                    iter_max, init_type, C.c_double(reweight), C.byref(e1), C.byref(e2),
                                    C.c_double(max_s_rho), C.c_uint(match_num_thresh),
                                    C.c_double(init_iter), _p(WX))
        return dict(F=F, V=V, W=W, RVel=RV, RW0=RW, W_X=WX, rel_err=e1.value, rel_err_score=e2.value)

    def try_vel_rot(self, old, X, reweight, procjf, match_thresh, s_rho_min, match_num_thresh, k_huber,
                    res_in):
        X = np.array(X, np.float64)
        pnum = (old.knum() + 3) & ~3
        res_in = np.ascontiguousarray(res_in, np.float64)
        assert len(res_in) == pnum
        res_out = np.full(pnum, np.nan)
        JtJ = np.zeros((6, 6))
        JtF = np.zeros(6)
        s = self.L.ref_try_vel_rot(self.h_, old.h_, _p(X), int(reweight), int(procjf),
                                   C.c_double(match_thresh), C.c_double(s_rho_min),
                                   C.c_uint(match_num_thresh), C.c_double(k_huber), _p(res_in),
                                   _p(res_out), _p(JtJ), _p(JtF))
        return s, JtJ, JtF, res_out

    def try_vel(self, old, V, match_thresh, s_rho_min, match_num_thresh, residuals, rw_dist, min_mod):
        V = np.array(V, np.float64)
        res = np.ascontiguousarray(residuals[:old.knum()], np.float64).copy()
        JtJ, JtF = np.zeros((3, 3)), np.zeros(3)
        self.L.ref_try_vel.restype = C.c_double
        s = self.L.ref_try_vel(self.h_, old.h_, _p(V), C.c_double(match_thresh), C.c_double(s_rho_min),
                               C.c_uint(match_num_thresh), _p(res), C.c_double(rw_dist), C.c_float(min_mod), _p(JtJ),
                               _p(JtF))
        return s, JtJ, JtF, res

    def minimizer_v(self, old, V, match_thresh, iter_max, s_rho_min, match_num_thresh, rw_dist, min_mod):
        V = np.array(V, np.float64)
        RV = np.zeros((3, 3))
        self.L.ref_minimizer_v.restype = C.c_double
        F = self.L.ref_minimizer_v(self.h_, old.h_, _p(V), _p(RV), C.c_double(match_thresh), iter_max,
                                   C.c_double(s_rho_min), C.c_uint(match_num_thresh), C.c_double(rw_dist),
                                   C.c_float(min_mod))
        return dict(F=F, V=V, RVel=RV)

    def ext_rot_vel(self, V, loc_unc, hub):
        V = np.array(V, np.float64)
        Wx, Rx, X = np.zeros((6, 6)), np.zeros((6, 6)), np.zeros(6)
        ok = self.L.ref_ext_rot_vel(self.h_, _p(V), _p(Wx), _p(Rx), _p(X), C.c_double(loc_unc), C.c_double(hub))
        return bool(ok), Wx, Rx, X

    def forward_match(self, new):
        return self.L.ref_forward_match(self.h_, new.h_)

    def rotate(self, R):
        R = np.ascontiguousarray(R, np.float64)
        self.L.ref_rotate(self.h_, _p(R))

    def directed_matching(self, old, V, RVel, BackRot, thr_mod, thr_ang, max_radius, loc_unc):
        V = np.ascontiguousarray(V, np.float64)
        RVel = np.ascontiguousarray(RVel, np.float64)
        BackRot = np.ascontiguousarray(BackRot, np.float64)
        kf = C.c_int(0)
        return self.L.ref_directed_matching(self.h_, old.h_, _p(V), _p(RVel), _p(BackRot), C.byref(kf),
                                            C.c_double(thr_mod), C.c_double(thr_ang),
                                            C.c_double(max_radius), C.c_double(loc_unc))

    def num_matches(self):
        return self.L.ref_num_matches(self.h_)

    def regularize(self, thresh):
        return self.L.ref_regularize(self.h_, C.c_double(thresh))

    def ekf(self, V, RVel, RW0, qabs, qrel, loc_unc):
        V = np.ascontiguousarray(V, np.float64)
        RVel = np.ascontiguousarray(RVel, np.float64)
        RW0 = np.ascontiguousarray(RW0, np.float64)
        self.L.ref_ekf(self.h_, _p(V), _p(RVel), _p(RW0), C.c_double(qabs), C.c_double(qrel),
                       C.c_double(loc_unc))

    def rescale(self, s_rho_min, match_num_min, re_escale):
        rkp = C.c_double(0)
        kp = self.L.ref_rescale(self.h_, C.byref(rkp), C.c_double(s_rho_min), C.c_uint(match_num_min),
                                int(re_escale))
        return kp, rkp.value


def undistort_rgb(cam, kc, rgb):
    """image_undistort(cam).undistort<true>(out, in) of the reference on one RGB24 frame."""
    rgb = np.ascontiguousarray(rgb, np.uint8)
    out = np.zeros_like(rgb)
    kc = np.ascontiguousarray(kc, np.float64)
    lib().ref_undistort_rgb(cam["w"], cam["h"], C.c_float(cam["ppx"]), C.c_float(cam["ppy"]), C.c_float(cam["zfx"]),
                            C.c_float(cam["zfy"]), _p(kc), _p(rgb), _p(out))
    return out


def bias_correct(X, Wx, Gb, Wb, Rg, Rb):
    """edge_tracker::BiasCorrect of the reference (in/out arrays)."""
    a = [np.ascontiguousarray(np.array(v, np.float64)) for v in (X, Wx, Gb, Wb)]
    Rg, Rb = np.ascontiguousarray(Rg, np.float64), np.ascontiguousarray(Rb, np.float64)
    lib().ref_bias_correct(_p(a[0]), _p(a[1]), _p(a[2]), _p(a[3]), _p(Rg), _p(Rb))
    return a


def so3_exp(w):
    w = np.ascontiguousarray(w, np.float64)
    R = np.zeros((3, 3))
    lib().ref_so3_exp(_p(w), _p(R))
    return R


def so3_ln(R):
    R = np.ascontiguousarray(R, np.float64)
    w = np.zeros(3)
    lib().ref_so3_ln(_p(R), _p(w))
    return w


OUTREC = np.dtype([("t", "f8"), ("Pos", "f8", 3), ("PoseLie", "f8", 3), ("Pose", "f8", 9), ("Vel", "f8", 3),
                   ("RotLie", "f8", 3), ("dtp0", "f8"), ("dtp1", "f8"), ("K", "f8"), ("Kp", "f8"),
                   ("s_rho_p", "f8"), ("kn", "i4"), ("matches", "i4"), ("est_ok", "i4"), ("p_id", "i4"),
                   ("Rot", "f8", 9), ("RKp", "f8"), ("dt", "f8")])


# a DT_NEEDED string that names librebvo_b200.so by an absolute path
_NEEDED_BY_PATH = re.compile(rb"/[^\0]*/librebvo_b200\.so\0")
_runnable = {}


def runnable(exe):
    """Path to start the oracle program `exe` (oracle/_ref/shim_driver, shim_rebvo) from.  A program linked against a
    librebvo_b200.so without a soname records the library by the absolute path of the tree it was built in: it does
    not start once that tree is gone, and would use that tree's library if it were not.  For such a program this
    returns a copy, under a temporary directory, whose DT_NEEDED entry names the library by file name (the string
    shrinks in place, NUL-padded) and which sits beside a link to this tree's rebvo_b200/, so that the program's
    $ORIGIN/../../rebvo_b200 rpath loads this tree's library.  Any other program is returned as it is."""
    if exe not in _runnable:
        with open(exe, "rb") as f:
            data = f.read()
        _runnable[exe] = exe
        if _NEEDED_BY_PATH.search(data):
            d = tempfile.mkdtemp(prefix="rebvo_oracle_")
            atexit.register(shutil.rmtree, d, True)
            os.symlink(os.path.join(os.path.dirname(HERE), "rebvo_b200"), os.path.join(d, "rebvo_b200"))
            os.makedirs(os.path.join(d, "oracle", "_ref"))
            out = os.path.join(d, "oracle", "_ref", os.path.basename(exe))
            with open(out, "wb") as f:
                f.write(_NEEDED_BY_PATH.sub(lambda m: b"librebvo_b200.so".ljust(len(m.group(0)), b"\0"), data))
            os.chmod(out, 0o755)
            _runnable[exe] = out
    return _runnable[exe]


def run_full_rebvo(frames_file, out_file, params=None, timeout=600, exe=None):
    """Level B: run the reference's whole 3-thread REBVO on a raw frame file (oracle/ref_driver.cpp).
    exe: another build of the same driver (oracle/_ref/shim_rebvo = the unmodified REBVO sources on the GPU library)."""
    import json
    import resource
    import subprocess

    def pre():
        # finite, large stack: the reference keeps O(27*8*K) byte VLAs on thread stacks (SURVEY.md section 7)
        resource.setrlimit(resource.RLIMIT_STACK, (1000000 * 1024, resource.RLIM_INFINITY))

    args = [runnable(exe or EXE), frames_file, out_file] + ["%s=%s" % (k, v if isinstance(v, str) else repr(v)) for k, v in (params or {}).items()]
    env = dict(os.environ)
    env["LD_LIBRARY_PATH"] = _blas_dir() + ":" + env.get("LD_LIBRARY_PATH", "")
    env.setdefault("OPENBLAS_NUM_THREADS", "1")
    r = subprocess.run(args, capture_output=True, text=True, timeout=timeout, preexec_fn=pre, env=env)
    if r.returncode != 0:
        raise RuntimeError("ref_rebvo failed: %s\n%s" % (r.returncode, r.stderr[-2000:]))
    line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
    info = json.loads(line)
    with open(out_file, "rb") as f:
        n, sz = np.frombuffer(f.read(8), np.int32)
        assert sz == OUTREC.itemsize, (sz, OUTREC.itemsize)
        rec = np.frombuffer(f.read(), OUTREC, count=n)
    return info, rec


def ref_params_from(p, **extra):
    """key=value arguments of oracle/ref_driver.cpp for a rebvo_b200.capi.Params (same parameter set on both sides)."""
    kv = dict(ZfX=p.cam.zfx, ZfY=p.cam.zfy, PPx=p.cam.ppx, PPy=p.cam.ppy, FPS=p.config_fps, Sigma0=p.Sigma0,
              KSigma=p.KSigma, DetectorPlaneFitSize=p.det.plane_fit_size, DetectorPosNegThresh=p.det.pos_neg_thresh,
              DetectorDoGThresh=p.det.dog_thresh, ReferencePoints=p.det.kl_ref, TrackPoints=p.TrackPoints,
              MaxPoints=p.det.kl_max, DetectorThresh=p.DetectorThresh, DetectorAutoGain=p.det.gain,
              DetectorMaxThresh=p.det.thresh_max, DetectorMinThresh=p.det.thresh_min,
              GlobalMatchThreshold=p.MatchThreshold, SearchRange=p.SearchRange, QCutOffNumBins=p.QCutOffNumBins,
              QCutOffQuantile=p.QCutOffQuantile, TrackerIterNum=p.TrackerIterNum,
              TrackerInitIterNum=p.TrackerInitIterNum, TrackerInitType=p.TrackerInitType,
              TrackerMatchThresh=p.TrackerMatchThresh, LocationUncertaintyMatch=p.LocationUncertaintyMatch,
              MatchThreshModule=p.MatchThreshModule, MatchThreshAngle=p.MatchThreshAngle,
              ReweigthDistance=p.ReweigthDistance, MatchNumThresh=p.MatchNumThresh, RegularizeThresh=p.RegularizeThresh,
              ReshapeQAbsolute=p.ReshapeQAbsolute, ReshapeQRelative=p.ReshapeQRelative,
              LocationUncertainty=p.LocationUncertainty, DoReScaling=p.DoReScaling)
    kv.update(extra)
    return kv


def trajectory_parity(rec, nav):
    """Pose / count agreement of a GPU run (rb_nav records) with the reference's run (OUTREC) on the same frames.
    Both trajectories come from identical inputs in the same camera frame: no alignment step (SURVEY.md 8(d))."""
    n = min(len(rec), len(nav))
    d = rec["Pos"][:n] - nav["Pos"][:n]
    e = np.sqrt((d ** 2).sum(1))
    return {"frames": int(n), "ate_m": float(np.sqrt((e ** 2).mean())), "max_pos_err_m": float(e.max()),
            "max_poselie_err_rad": float(np.abs(rec["PoseLie"][:n] - nav["PoseLie"][:n]).max()),
            "path_length_m": float(np.linalg.norm(np.diff(rec["Pos"][:n], axis=0), axis=1).sum()),
            "kn_equal": bool(np.array_equal(rec["kn"][:n], nav["kn"][:n])),
            "matches_equal": bool(np.array_equal(rec["matches"][1:n], nav["matches"][1:n])),
            "estimation_ok_equal": bool(np.array_equal(rec["est_ok"][1:n] != 0, nav["estimation_ok"][1:n] != 0)),
            "first_kn_mismatch": int(np.nonzero(rec["kn"][:n] != nav["kn"][:n])[0][0])
            if not np.array_equal(rec["kn"][:n], nav["kn"][:n]) else -1}
