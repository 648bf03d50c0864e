#!/usr/bin/env python
"""bench.py -- frames/s of the REBVO edge pipeline (detect + track + map, pose out) on B200.

Workload (BASELINE.json configs[1]): EuRoC MH_01-like 752x480 replay, IMU off, parameters of
app/rebvorun/GlobalConfig_EuRoC_2.txt with TrackerInitType=2 (12 TryVelRot evaluations per frame).  No dataset
is available offline, so the stream is the seeded two-layer parallax generator of rebvo_b200/synth.py
(SURVEY.md section 8(d) fallback).  One "step" = one batch of `--batch` consecutive frames pushed through
rb_pipeline_push*: batched scale space for the batch, then detection + tracking + mapping frame by frame (the
tracker is a recurrence over frames).

  value : whole-job frames/s with the RGB frames already resident in HBM (rb_pipeline_push_dev)
  e2e   : the same through the C ABI with HOST (pinned) frame buffers, H2D of the frames and D2H of the nav
          records inside the timed region
  --impl reference : the reference's own three-thread CPU REBVO (oracle/_ref/ref_rebvo, unmodified sources)
          on a bounded sample of the same stream, host cores only.

Multi-GPU (torchrun, one rank per GPU): the tracker does not shard (SURVEY.md 8(e)) -> independent replicas,
one sequence per rank, no data-path collective; NCCL is used for the barrier and the max-over-ranks time.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "frames/sec @752x480 EuRoC replay (synthetic stand-in), detect+track+map; pose ATE vs reference in `parity`"
WORKLOAD = ("configs[1]: EuRoC MH_01-like 752x480 full replay, 1xB200 per sequence, IMU off (pure edge VO), UseUndistort=1 with "
            "the EuRoC rad-tan coefficients in both arms; synthetic two-layer parallax stream seed 7")


def rank_info():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


TUM_CAM = dict(w=640, h=480, zfx=525.0, zfy=525.0, ppx=320.0, ppy=240.0)
METRIC5 = "frames/sec @640x480 TUM desk parameters (synthetic stand-in), detect+track+map; pose ATE vs reference in `parity`"
WORKLOAD5 = ("configs[4]: TUM fr2_desk-like 640x480 replay, app/rebvorun/GlobalConfig_desk.txt parameters (Sigma0 1.7818, auto-"
             "threshold gain 1e-6, SearchRange 20, TrackerIterNum 10 = 17 TryVelRot evaluations per frame, MatchNumThresh 4); "
             "synthetic two-layer parallax stream seed 21")


METRIC3 = ("frames/sec @752x480 EuRoC replay with IMU fusion (ImuMode=2, synthetic stand-in), detect+track+map+scale filter; "
           "pose ATE vs reference in `parity`")
WORKLOAD3 = ("configs[2]: EuRoC V1_02-like 752x480 replay with ImuGrabber csv fusion (IMUMode=2), 1xB200; synthetic two-layer "
             "parallax stream seed 7 + synthetic 200 Hz IMU (gyro bias 0.02 rad/s, noise 1.7e-4); UseUndistort=1 in both arms")
IMU_BASE_N = 160


# GlobalConfig_EuRoC_2.txt:64-68,73: the EuRoC configurations run UseUndistort=1 with these rad-tan coefficients
EUROC_KC = (-0.28340811, 0.07395907, 0.0, 0.00019359, 1.76187114e-05)


def undistort_of(config):
    """distortion coefficients both arms undistort with (None: UseUndistort=0, the desk / synthetic configurations)"""
    return EUROC_KC if config in (2, 3) else None


def stream_setup(config):
    """camera, parameters, metric / workload strings of the single-sequence bench configurations"""
    from rebvo_b200 import capi, synth
    if config == 3:
        return synth.EUROC, capi.default_params(synth.EUROC), METRIC3, WORKLOAD3, 7
    if config == 5:
        p = capi.default_params(TUM_CAM, Sigma0=1.7818, kl_max=25000, kl_ref=15000, gain=1e-6, thresh_max=0.05,
                                thresh_min=0.03, SearchRange=20, TrackerIterNum=10, TrackerMatchThresh=1.0, MatchNumThresh=4,
                                ReshapeQRelative=1e-2, kl_capacity=25000)
        return TUM_CAM, p, METRIC5, WORKLOAD5, 21
    return synth.EUROC, capi.default_params(synth.EUROC), METRIC, WORKLOAD, 7


def make_stream(seed, total, base_n=160, cam=None):
    """total frames of a continuous sequence built from base_n rendered frames walked back and forth."""
    from rebvo_b200 import synth
    cam = cam or synth.EUROC
    seq = synth.Sequence(w=cam["w"], h=cam["h"], seed=seed, zf=cam["zfx"])
    base_n = min(base_n, total)
    _, base = seq.frames(base_n)
    period = max(1, 2 * (base_n - 1))
    idx = np.arange(total) % period
    idx = np.where(idx < base_n, idx, period - idx)
    ts = np.arange(total) / 20.0
    return ts, base, idx


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.p = [], None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                      stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append((time.time(), line.strip()))

    def mark(self):
        return time.time()

    def summary(self, t0, t1):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm, mx, reasons = [], None, set()
        for t, line in self.rows:
            if t < t0 or t > t1 + 0.15:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}

    def stop(self):
        if self.p:
            self.p.terminate()


# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture
# (profiles/r1_summary.md section 3, 64-frame batch = the default bench batch)
TRAFFIC = {"k_rowscan_ring<avg>": 3.19e8,   # 307-331 MB over the two launches of a 64-frame batch (round 1)
           "k_rowscan_tma_avg": 3.31e8,     # 188.9 MB read + 142.2 MB written (profiles/r2_summary.md section 4)
           "k_rowscan_tma_plain": 1.385e8,  # 94.4 MB read + 44.1 MB written (the rest of the 92 MB written is still in L2)
           "k_minimizer_cluster": 2.43e6}   # profiles/r2_summary.md section 3 (operands / residuals in shared memory, gathers in L1)


def peak_gbs():
    return peaks()[0]


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def dump_outputs(path, nav):
    """--dump-outputs: every field of the nav records the timed path returned for its last step, one <field>.npy per
    field (float32 fields as they are, the others as float64, exact for the int32 counters), so that two builds run
    with the same arguments can be compared output for output."""
    os.makedirs(path, exist_ok=True)
    for name in nav.dtype.names:
        a = nav[name]
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a, np.float32 if a.dtype == np.float32 else np.float64))


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def run_reference(frames_file_dir, ts, base, idx, n_frames, warm_frames, affinity=True, gpu_params=None, imu=None, kc=None):
    """The reference's own CPU implementation (3 pipeline threads) on n_frames of the stream."""
    from oracle import refapi
    from rebvo_b200 import synth
    path = os.path.join(frames_file_dir, "rebvo_b200_bench_frames_%d.bin" % os.getpid())
    synth.write_frames_file(path, ts[:n_frames], base[idx[:n_frames]])
    ncpu = os.cpu_count() or 1
    params = refapi.ref_params_from(gpu_params) if gpu_params is not None else {}
    params["Warmup"] = warm_frames
    csv = None
    if imu is not None:   # config 3: the reference reads the same samples through ImuGrabber::LoadDataSet
        csv = path + ".imu.csv"
        synth.write_imu_csv(csv, imu)
        params.update(ImuMode=2, ImuFile=csv, ImuTimeScale=1, InitBias=1, InitBiasFrameNum=5)
    if kc is not None:
        params.update(UseUndistort=1, KcR2=kc[0], KcR4=kc[1], KcR6=kc[2], KcP1=kc[3], KcP2=kc[4])
    if affinity and ncpu >= 3:
        params.update(SetAffinity=1, CPU0=0, CPU1=1, CPU2=2)
    try:
        info, rec = refapi.run_full_rebvo(path, path + ".out", params, timeout=1800)
    finally:
        for f in (path, path + ".out", csv):
            if f and os.path.exists(f):
                os.remove(f)
    return info, rec


def bench_reference(args):
    rank, local_rank, world = rank_info()
    if rank != 0:
        return
    from oracle import refapi
    if not os.path.exists(refapi.EXE):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/ref_rebvo not built (reference sources absent)"}))
        return
    per = max(20, min(60, 600 // (args.steps + args.warmup)))
    total = per * (args.steps + args.warmup) + 2
    if args.config == 4:   # same 1280x960 stream and parameters as the GPU arm's sequence 0
        from rebvo_b200 import capi
        cam, params, metric, workload = BIG_CAM, big_params(capi), METRIC4, WORKLOAD4 % args.seqs
        per = max(8, min(16, 160 // (args.steps + args.warmup)))
        total = per * (args.steps + args.warmup) + 2
        base = big_stream(100, total)
        idx = walk_index(total, len(base), 0)
        ts = np.arange(total) / 20.0
    else:
        cam, params, metric, workload, seed0 = stream_setup(args.config)
        ts, base, idx = make_stream(seed0, total, cam=cam)
    imu = None
    if args.config == 3:
        from rebvo_b200 import synth
        seq = synth.Sequence(w=cam["w"], h=cam["h"], seed=seed0, zf=cam["zfx"])
        imu = synth.imu_samples_walk(seq, total, min(IMU_BASE_N, total))
    info, rec = run_reference(tempfile.gettempdir(), ts, base, idx, total, per * args.warmup, gpu_params=params, imu=imu,
                              kc=undistort_of(args.config))
    fps = info["fps"]
    ncpu = os.cpu_count() or 1
    out = {"metric": metric, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": 1e3 * per / fps, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32 scale space/detector + f64 tracker/EKF", "data": "synthetic",
           "impl": "reference",
           "config": {"workload": workload, "frames_per_step": per, "note": "bounded sample of the bench stream"},
           "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": 3, "kind": "reference", "cpu_model": cpu_model(),
                            "sample": "%d frames (%d timed) through the unmodified 3-thread REBVO, %d host cpus visible"
                            % (total, info["timed_callbacks"], ncpu),
                            "mean_dtp0_ms": info["mean_dtp0_ms"], "mean_dtp1_ms": info["mean_dtp1_ms"]},
           "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


def bench_ours(args):
    import torch
    from rebvo_b200 import multi
    rank, local_rank, world = multi.rank_info()
    dist = None
    if world > 1:
        torch.cuda.set_device(local_rank)
        dist = multi.init("nccl", device=torch.device("cuda", local_rank))
    dev = local_rank if world > 1 else 0
    torch.cuda.set_device(dev)
    from rebvo_b200 import capi, synth
    B, K, W = args.batch, args.steps, args.warmup
    total = B * (K + W)
    cam, params, metric, workload, seed0 = stream_setup(args.config)
    ts, base, idx = make_stream(multi.stream_seed(rank) + (seed0 - 7), total, cam=cam)
    imu = None
    if args.config == 3:   # IMU samples of the walked camera path; every pipeline of this run gets them
        seq = synth.Sequence(w=cam["w"], h=cam["h"], seed=multi.stream_seed(rank), zf=cam["zfx"])
        imu = synth.imu_samples_walk(seq, total, min(IMU_BASE_N, total))
    h, w = cam["h"], cam["w"]
    fbytes = h * w * 3
    # host (pinned) and device copies of the whole stream, batch-contiguous
    host = torch.empty((total, h, w, 3), dtype=torch.uint8, pin_memory=True)
    host.numpy()[:] = base[idx]
    devbuf = host.to("cuda:%d" % dev)
    torch.cuda.synchronize()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(dev)
    # ---------------- value: frames resident in HBM ----------------------------------------------------
    kc = undistort_of(args.config)

    def new_pipeline():
        q = capi.Pipeline(params, max_batch=B, device=dev)
        if kc is not None:
            q.set_undistort(kc)
        return q
    pl = new_pipeline()
    if imu is not None:
        pl.set_imu(imu, capi.default_imu_params(InitBias=1, InitBiasFrameNum=5))
    navs = []
    for s in range(W):
        navs.append(pl.push_dev(devbuf[s * B].data_ptr(), ts[s * B:(s + 1) * B]))
    barrier()
    l0 = pl.launches()
    c0 = sampler.mark()
    pl.event_record(0)
    for s in range(W, W + K):
        navs.append(pl.push_dev(devbuf[s * B].data_ptr(), ts[s * B:(s + 1) * B]))
    pl.event_record(1)
    barrier()
    c1 = sampler.mark()
    t_dev_ms = pl.event_elapsed(0, 1)
    launches = pl.launches() - l0
    nav_dev = np.concatenate(navs)
    # ---------------- roofline of the scale-space passes (same workspace, same batch) --------------------
    passes = {}
    # (names of the kernels the library dispatches to by default; the environment switches select the older versions)
    row_tma = os.environ.get("REBVO_B200_ROW_TMA", "1") != "0" and w % 4 == 0
    rs = "k_rowscan_ring" if os.environ.get("REBVO_B200_ROWSCAN", "2") == "2" else "k_rowscan"
    rs_plain, rs_avg = ("k_rowscan_tma_plain", "k_rowscan_tma_avg") if row_tma else (rs + "<plain>", rs + "<avg>")
    blur = "k_blur_dog_tma" if os.environ.get("REBVO_B200_BLUR_TMA", "1") != "0" and w % 4 == 0 else "k_blur_dog"
    peak_now = peak_gbs()
    gray = "k_undistort_gray" if kc is not None else "k_rgb2gray"
    for pid, name in ((5 if kc is not None else 4, gray), (0, rs_plain), (1, rs_avg), (2, "k_colscan_pipe"), (3, blur)):
        ms, by = pl.bench_pass(pid, B, 20)
        passes[name] = {"ms_per_launch": ms, "bytes_per_launch": by, "gbs": by / (ms * 1e-3) / 1e9,
                        "frac": by / (ms * 1e-3) / 1e9 / peak_now}
    pl.close()
    # ---------------- e2e: host buffers through the C ABI ------------------------------------------------
    pl2 = new_pipeline()
    if imu is not None:
        pl2.set_imu(imu, capi.default_imu_params(InitBias=1, InitBiasFrameNum=5))
    navs2 = []
    for s in range(W):
        navs2.append(pl2.push(host[s * B].data_ptr(), ts[s * B:(s + 1) * B]))
    barrier()
    pl2.event_record(0)
    for s in range(W, W + K):
        navs2.append(pl2.push(host[s * B].data_ptr(), ts[s * B:(s + 1) * B]))
    pl2.event_record(1)
    barrier()
    t_e2e_ms = pl2.event_elapsed(0, 1)
    nav_e2e = np.concatenate(navs2)
    pl2.close()
    # ---------------- e2e with the per-frame host mirror (SURVEY 8(d): the 168-byte KeyLine AoS D2H, reported separately) ----
    mirror = None
    if rank == 0 and imu is None:
        mirror = {}
        # raw D2H rate of this box (one 256 MB pinned copy): what bounds the 168-byte mirror
        hb = torch.empty(256 << 20, dtype=torch.uint8, pin_memory=True)
        db = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:%d" % dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        hb.copy_(db, non_blocking=True)
        torch.cuda.synchronize()
        e0.record()
        hb.copy_(db, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        d2h_gbs = (256 << 20) / (e0.elapsed_time(e1) * 1e-3) / 1e9
        del hb, db
        for mode, key, rec in ((1, "keyline_168B", capi.KEYLINE.itemsize), (2, "net_keyline_15B", 15)):
            pl4 = new_pipeline()
            pl4.set_mirror(mode)
            for s in range(W):
                pl4.push(host[s * B].data_ptr(), ts[s * B:(s + 1) * B])
            pl4.event_record(0)
            mbytes = 0
            for s in range(W, W + K):
                navm = pl4.push(host[s * B].data_ptr(), ts[s * B:(s + 1) * B])
                mbytes += int(navm["kn"].sum()) * rec
            pl4.event_record(1)
            t_m = pl4.event_elapsed(0, 1)
            pl4.close()
            mirror[key] = {"value": K * B / (t_m * 1e-3), "unit": "frames/s", "ms_per_step": t_m / K,
                           "d2h_mirror_bytes_per_step": mbytes / K, "d2h_gbs": mbytes / (t_m * 1e-3) / 1e9}
        mirror["d2h_copy_peak_gbs"] = d2h_gbs
        mirror["what"] = ("e2e plus every frame's edge map in pinned host memory (rb_pipeline_set_mirror: packed after the "
                          "frame's map update, written to mapped host memory while the next frames are tracked): as the reference's 168-byte KeyLine array, and as the "
                          "15-byte net_keyline records its third thread sends")
    # ---------------- where the step goes: in-situ stage profile (eager launches, one stream, CUDA events) ---------
    stage_us = None
    if rank == 0 and imu is None:   # (the IMU-mode frame loop is host-driven: no per-stage device profile)
        os.environ["REBVO_B200_STAGE_PROF"] = "1"
        try:
            pl3 = new_pipeline()
            for s in range(min(3, K + W)):
                pl3.push_dev(devbuf[s * B].data_ptr(), ts[s * B:(s + 1) * B])
            stage_us, _ = pl3.stage_profile()
            pl3.close()
        finally:
            del os.environ["REBVO_B200_STAGE_PROF"]
    sampler.stop()
    clocks = sampler.summary(c0, c1)
    same = bool(np.array_equal(nav_dev["Pos"], nav_e2e["Pos"]))

    t_max, t_e2e_max = multi.max_over_ranks(dist, [t_dev_ms, t_e2e_ms], device="cuda:%d" % dev)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    value = multi.aggregate_fps(K * B, world, t_max)
    e2e = multi.aggregate_fps(K * B, world, t_e2e_max)
    peak, peak_src = peaks()
    # launches of each scale-space pass in one step (rb_dog_build_batch: gray, one plain row pass and one column pass over
    # B images, then per box stage an averaged row pass + a column pass over 2B images, then the blur/DoG pass); the
    # timed column pass is the 2B-image one, the B-image one counts half
    per_step = {gray: 1, rs_plain: 1, rs_avg: 2, "k_colscan_pipe": 2.5, blur: 1}
    dog_ms = sum(passes[k]["ms_per_launch"] * n for k, n in per_step.items())
    # ---- roofline of the TIME-dominant kernel: Minimizer_RV (one launch per frame).  Algorithmic bytes per launch =
    # SURVEY.md 8(d) tryvelrot_bytes = E * (K0 * 104 + 224), E = TryVelRot evaluations (2*(init_iter+1) + 1 + iter), K0 = old
    # keylines; duration = CUDA events around the kernel in the eager stage-profile pass of this same run.
    kn_mean = float(nav_dev["kn"].mean())
    evals = (2 * (params.TrackerInitIterNum + 1) if params.TrackerInitType not in (0, 1) else 0) + 1 + params.TrackerIterNum
    tvr_bytes = evals * (kn_mean * 104.0 + 224.0)
    min_us = stage_us["minimizer"] if stage_us else None
    min_gbs = tvr_bytes / (min_us * 1e-6) / 1e9 if min_us else None
    N = h * w
    stage_gbs = {}
    if stage_us:
        # field: 8N + (20 + 2r*8) K_f (K_f ~ TrackPoints); mapper: rotate 64 K0 + fwdmatch 24 K0 + 80 M + dmatch (40 K + 128 M)
        # + regularize 96 K + ekf 84 M + rescale 5*32 K (mask probes / candidates of the search are not counted: lower bound)
        m_mean = float(nav_dev["matches"][1:].mean())
        field_b = 8.0 * N + (20 + 2 * params.SearchRange * 8) * min(kn_mean, params.TrackPoints)
        mapper_b = 64 * kn_mean + 24 * kn_mean + 80 * m_mean + 40 * kn_mean + 128 * m_mean + 96 * kn_mean + 84 * m_mean + 160 * kn_mean
        mapper_us = sum(stage_us[k] for k in ("fwdmatch+rotate", "directed_match", "regularize+ekf", "rescale"))
        stage_gbs = {"minimizer": {"us": min_us, "algorithmic_bytes": tvr_bytes, "gbs": min_gbs, "frac": min_gbs / peak_gbs()},
                     "quantile+field": {"us": stage_us["quantile+field"], "algorithmic_bytes": field_b,
                                        "gbs": field_b / (stage_us["quantile+field"] * 1e-6) / 1e9},
                     "mapper": {"us": mapper_us, "algorithmic_bytes_lower_bound": mapper_b,
                                "gbs": mapper_b / (mapper_us * 1e-6) / 1e9}}
    dom = min(passes, key=lambda k: passes[k]["gbs"])   # the scale-space pass furthest from the roofline
    roof = {"bound": "hbm", "kernel": "k_minimizer_cluster (Minimizer_RV, one launch per frame)",
            "achieved": min_gbs, "peak": peak, "unit": "GB/s", "frac": (min_gbs / peak) if min_gbs else None,
            "traffic": TRAFFIC.get("k_minimizer_cluster"), "peak_source": peak_src,
            "algorithmic_bytes_per_launch": tvr_bytes, "ms_per_launch": (min_us * 1e-3) if min_us else None,
            "evaluations_per_launch": evals,
            "note": "time-dominant kernel of the step. It is LATENCY-bound, not bandwidth-bound: its rounds are strictly "
                    "dependent (the pose of an evaluation is the LM step on the sums over all keylines of the previous one); "
                    "the bandwidth fraction is reported because SURVEY 8(d) defines the metric, see DESIGN.md section 4 for "
                    "the per-round breakdown. The kernels that carry the step's HBM traffic are under scale_space.",
            "stages": stage_gbs,
            "scale_space": {"kernel": dom, "achieved": passes[dom]["gbs"], "frac": passes[dom]["gbs"] / peak,
                            "traffic": TRAFFIC.get(dom), "all_passes": passes,
                            "share_of_step": dog_ms / (t_max / K) if t_max > 0 else None,
                            "whole_scale_space_gbs": 103.0 * N * B / (dog_ms * 1e-3) / 1e9,
                            "whole_scale_space_frac": 103.0 * N * B / (dog_ms * 1e-3) / 1e9 / peak},
            "stage_us_per_frame_eager": stage_us}
    cpu = None
    parity = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            n = min(620, total)
            info, rec = run_reference(tempfile.gettempdir(), ts, base, idx, n, 20, gpu_params=params, imu=imu,
                                      kc=undistort_of(args.config))
            cpu = {"value": info["fps"], "unit": "frames/s", "cores": 3, "kind": "reference", "cpu_model": cpu_model(),
                   "sample": "first %d frames of the bench stream (20 warm-up) through the unmodified 3-thread REBVO "
                             "built from the reference sources; %d host cpus visible" % (n, os.cpu_count() or 1),
                   "mean_dtp0_ms": info["mean_dtp0_ms"], "mean_dtp1_ms": info["mean_dtp1_ms"]}
            from oracle import refapi
            parity = refapi.trajectory_parity(rec, nav_dev)
            parity["vs"] = "reference CPU build, same %d frames of the bench stream, same parameters" % n
            parity["e2e_arm"] = refapi.trajectory_parity(rec, nav_e2e)
            # level A (BASELINE.md section 4): the reference's functions, one thread, stage by stage, on a frame pair of this stream,
            # beside this library's per-frame stage times of the same run (CUDA events, eager launches)
            from oracle import level_a
            la_cfg = level_a.TUM if args.config == 5 else level_a.EUROC
            try:   # (the reference keeps O(27 * 8 * K) bytes of VLAs on the caller's stack)
                import resource
                resource.setrlimit(resource.RLIMIT_STACK, (min(1 << 30, resource.getrlimit(resource.RLIMIT_STACK)[1])
                                                           if resource.getrlimit(resource.RLIMIT_STACK)[1] != resource.RLIM_INFINITY
                                                           else 1 << 30, resource.getrlimit(resource.RLIMIT_STACK)[1]))
            except (ImportError, ValueError, OSError):
                pass
            la = level_a.stage_table(la_cfg, np.ascontiguousarray(base[idx[10]]), np.ascontiguousarray(base[idx[11]]), reps=5)
            cpu["level_a"] = {"threads": 1, "config": la_cfg["name"], "ms_per_frame": la,
                              "what": "unmodified reference functions (oracle/_ref/libref_mtrack.so), median of 5 runs of the "
                                      "per-frame chain on frames 10/11 of the bench stream, old map seeded with rho = 1",
                              "gpu_us_per_frame_eager": stage_us}
        except Exception as e:  # the oracle is test infrastructure; its absence must not break the bench
            cpu = {"value": None, "unit": "frames/s", "cores": 0, "kind": "reference", "sample": "unavailable: %r" % (e,)}
    ok = nav_dev["estimation_ok"]
    out = {"metric": metric, "value": value, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
           "ms_per_step": t_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32 scale space/detector + f64 tracker/EKF", "data": "synthetic",
           "config": {"workload": workload, "frames_per_step": B, "sequences": world, "parallelism": "replicas x%d" % world,
                      "l2": "inputs larger than L2: per-step working set %.0f MB (RGB %.0f MB + scale-space planes)"
                            % (B * (3 + 32) * h * w / 1e6, B * fbytes / 1e6),
                      "keylines_mean": float(nav_dev["kn"].mean()), "tracked_ok_frac": float(ok[1:].mean()),
                      "dev_vs_e2e_identical_pose": same},
           "clocks": clocks,
           "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": B * fbytes,
                   "d2h_bytes_per_step": B * capi.NAV.itemsize, "ms_per_step": t_e2e_max / K},
           "e2e_with_mirror": mirror,
           "gpu_launches": int(launches), "gpu_launches_per_frame": launches / (K * B),
           "parity": parity, "roofline": roof, "cpu_baseline": cpu}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, navs[-1])
    print(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------------
# BASELINE.json configs[3]: synthetic 1280x960, ~30 k keylines, 8 frames per batch, several independent sequences per GPU
# (each its own rb_pipeline: own context, streams and CUDA graphs; one-cluster minimiser so that co-residency is
# guaranteed whatever the other pipelines do) x N GPUs.  Throughput test: frames of all sequences / device time.
# ---------------------------------------------------------------------------------------------------------------------
BIG_CAM = dict(w=1280, h=960, zfx=780.0, zfy=778.0, ppx=640.5, ppy=479.25)
WORKLOAD4 = ("configs[3]: synthetic 1280x960 stream, ~30k keylines per frame (ReferencePoints=30000, MaxPoints=40000), "
             "batches of 8 frames, %d independent sequences per GPU")
METRIC4 = "frames/sec @1280x960 synthetic 30k-keyline streams, 8-frame batches, several sequences per GPU, detect+track+map"


def big_params(capi):
    return capi.default_params(BIG_CAM, kl_ref=30000, kl_max=40000, TrackPoints=24000, kl_capacity=40000)


def big_stream(seed, total, base_n=24):
    from rebvo_b200 import synth
    seq = synth.Sequence(w=BIG_CAM["w"], h=BIG_CAM["h"], seed=seed, zf=BIG_CAM["zfx"], nrect_bg=1500, nrect_fg=200)
    base_n = min(base_n, total)
    _, base = seq.frames(base_n)
    return base


def walk_index(total, base_n, start):
    period = max(1, 2 * (base_n - 1))
    idx = (np.arange(total) + start) % period
    return np.where(idx < base_n, idx, period - idx)


def bench_config4(args):
    import threading as th
    import torch
    from rebvo_b200 import multi
    rank, local_rank, world = multi.rank_info()
    dist = None
    if world > 1:
        torch.cuda.set_device(local_rank)
        dist = multi.init("nccl", device=torch.device("cuda", local_rank))
    dev = local_rank if world > 1 else 0
    torch.cuda.set_device(dev)
    os.environ.setdefault("REBVO_B200_MIN_G", "1")       # one cluster per minimisation: pipelines share the GPU
    os.environ.setdefault("REBVO_B200_MIN_KPC", "2528")  # 40 k keylines per map in shared memory
    from rebvo_b200 import capi
    S, B, K, W = args.seqs, 8, args.steps, args.warmup
    total = B * (K + W)
    base = big_stream(100 + rank, total)
    base_n = len(base)
    h, w = BIG_CAM["h"], BIG_CAM["w"]
    fbytes = h * w * 3
    ts = np.arange(total) / 20.0
    params = big_params(capi)
    host, devb, pls = [], [], []
    for s in range(S):   # sequence s walks the rendered frames from its own starting point
        idx = walk_index(total, base_n, 3 * s)
        hb = torch.empty((total, h, w, 3), dtype=torch.uint8, pin_memory=True)
        hb.numpy()[:] = base[idx]
        host.append(hb)
        devb.append(hb.to("cuda:%d" % dev))
        pls.append(capi.Pipeline(params, max_batch=B, device=dev))
    torch.cuda.synchronize()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def run(on_device):
        navs = [[] for _ in range(S)]
        errs = []

        def worker(s, lo, hi):
            try:
                for k in range(lo, hi):
                    sl = slice(k * B, (k + 1) * B)
                    if on_device:
                        navs[s].append(pls[s].push_dev(devb[s][k * B].data_ptr(), ts[sl]))
                    else:
                        navs[s].append(pls[s].push(host[s][k * B].data_ptr(), ts[sl]))
            except Exception as e:   # noqa
                errs.append(e)

        def phase(lo, hi):
            thr = [th.Thread(target=worker, args=(s, lo, hi)) for s in range(S)]
            for t in thr:
                t.start()
            for t in thr:
                t.join()
            if errs:
                raise errs[0]

        for p in pls:
            p.reset()
        phase(0, W)
        barrier()
        l0 = sum(p.launches() for p in pls)
        pls[0].event_record(0)
        phase(W, W + K)
        for p in pls:
            p.event_record(1)
        barrier()
        ms = max(p.event_elapsed_from(pls[0], 0, 1) for p in pls)
        return ms, sum(p.launches() for p in pls) - l0, [np.concatenate(n) for n in navs]

    sampler = ClockSampler(dev)
    c0 = sampler.mark()
    t_dev_ms, launches, nav_dev = run(True)
    c1 = sampler.mark()
    t_e2e_ms, _, nav_e2e = run(False)
    sampler.stop()
    clocks = sampler.summary(c0, c1)
    t_max, t_e2e_max = multi.max_over_ranks(dist, [t_dev_ms, t_e2e_ms], device="cuda:%d" % dev)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    frames = S * K * B
    value = multi.aggregate_fps(frames, world, t_max)
    e2e = multi.aggregate_fps(frames, world, t_e2e_max)
    cpu = None
    parity = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            from oracle import refapi
            from rebvo_b200 import synth
            n = min(40, total)
            idx = walk_index(total, base_n, 0)
            path = os.path.join(tempfile.gettempdir(), "rebvo_b200_bench4_%d.bin" % os.getpid())
            synth.write_frames_file(path, ts[:n], base[idx[:n]])
            kv = refapi.ref_params_from(params, Warmup=8)
            if (os.cpu_count() or 1) >= 3:
                kv.update(SetAffinity=1, CPU0=0, CPU1=1, CPU2=2)
            try:
                info, rec = refapi.run_full_rebvo(path, path + ".out", kv, timeout=1800)
            finally:
                for f in (path, path + ".out"):
                    if os.path.exists(f):
                        os.remove(f)
            cpu = {"value": info["fps"], "unit": "frames/s", "cores": 3, "kind": "reference", "cpu_model": cpu_model(),
                   "sample": "%d frames of sequence 0 (8 warm-up) through the unmodified 3-thread REBVO" % n}
            parity = refapi.trajectory_parity(rec, nav_dev[0])
        except Exception as e:
            cpu = {"value": None, "unit": "frames/s", "cores": 0, "kind": "reference", "sample": "unavailable: %r" % (e,)}
    out = {"metric": METRIC4, "value": value, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
           "ms_per_step": t_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32 scale space/detector + f64 tracker/EKF", "data": "synthetic",
           "config": {"workload": WORKLOAD4 % S, "frames_per_step": S * B, "sequences_per_gpu": S, "sequences": S * world,
                      "parallelism": "replicas x%d, %d pipelines per GPU" % (world, S),
                      "l2": "inputs larger than L2: %.0f MB of frames + scale-space planes in flight per step" % (S * B * 38 * h * w / 1e6),
                      "keylines_mean": float(np.mean([n["kn"].mean() for n in nav_dev])),
                      "tracked_ok_frac": float(np.mean([n["estimation_ok"][1:].mean() for n in nav_dev])),
                      "minimizer": "one 16-CTA cluster per sequence (REBVO_B200_MIN_G=1)",
                      "dev_vs_e2e_identical_pose": bool(all(np.array_equal(a["Pos"], b["Pos"]) for a, b in zip(nav_dev, nav_e2e)))},
           "clocks": clocks,
           "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": S * B * fbytes,
                   "d2h_bytes_per_step": S * B * capi.NAV.itemsize, "ms_per_step": t_e2e_max / K},
           "gpu_launches": int(launches), "gpu_launches_per_frame": launches / frames,
           "parity": parity, "roofline": None, "cpu_baseline": cpu}
    if args.dump_outputs:   # leading axis: the sequence
        dump_outputs(args.dump_outputs, np.stack([n[-B:] for n in nav_dev]))
    print(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5], help="BASELINE.json configs index + 1 (2: 752x480 EuRoC-like replay, 3: the same with IMU fusion, 4: 1280x960 multi-sequence, 5: 640x480 TUM desk parameters)")
    ap.add_argument("--seqs", type=int, default=8, help="config 4: independent sequences per GPU")
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of this library's pipeline, not of --impl reference")
    if args.impl == "reference":
        bench_reference(args)
    elif args.config == 4:
        bench_config4(args)
    else:
        bench_ours(args)


if __name__ == "__main__":
    main()
