#!/usr/bin/env python
"""bench.py -- headline benchmark of the two hot paths (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of FeatureTracker::trackImage over one batch of FRAMES_PER_STEP = 100 consecutive 640x480 RGB-D frames
of a synthetic stream with 150 features (BASELINE.json configs[1], "C2"), submitted as ONE library call
(gf_tracker_track_batch: two frames in flight).  Rank r tracks its own stream (seed r): weak scaling, no data-path
collective (SURVEY 8e); the timed region of K steps is bracketed by barrier + synchronize and the maximum over ranks is
reported.

  value         frames/s with the frames already resident in HBM (device pointers)
  e2e           frames/s through the same call with pinned HOST frames: the H2D copy of gray + depth and the D2H copy of
                the observations of every frame are inside the timed region
  roofline      of the dominant kernel (k_track: forward + reverse pyramidal LK), algorithmic bytes / duration
  cpu_baseline  the reference's CPU path on this box's host cores (bounded sample): its three OpenCV calls (cv2 4.13)
                + its glue in C (oracle/fe_oracle.py::FeatureTrackerOracleFast); both the whole call and the OpenCV part
  streams       N=1: several independent trackers on one GPU (1/2/4/8 host threads): the multi-stream figure of SURVEY 8(d)
  configs       N=1: C3 (300 features) and C4 front end (1280x720, 500 features) lines; N>1: the C5 line (300 features / stream)
  ba            N=1: sliding-window solves/s through gf_ba_solve next to the CPU oracle, roofline against the measured
                FP64 rate of the device, marginalisation times

--impl reference times the reference's CPU path: the reference cannot be compiled here (ROS / Eigen / Ceres / OpenCV C++
absent), so this is the restatement on the same three OpenCV entry points (kind "port"), all host threads.

--dump-outputs DIR writes, as float64 .npy files, what the last timed step of the headline (device-resident) run returned to
its caller: the observations, inlier masks and counters of its FRAMES_PER_STEP frames (rank 0's stream).  The inputs depend
only on the arguments, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FRAMES_PER_STEP = 100
WORKLOADS = {
    "C2": dict(w=640, h=480, max_cnt=150, min_dist=30, ring=160,
               name="C2: synthetic 640x480 RGB-D stream, 150 features, min_dist 30, flow_back 1 (BASELINE.json configs[1])"),
    "C3": dict(w=640, h=480, max_cnt=300, min_dist=20, ring=160,
               name="C3/C5 front end: synthetic 640x480 RGB-D stream, 300 features, min_dist 20 (BASELINE.json configs[2], [4])"),
    "C4": dict(w=1280, h=720, max_cnt=500, min_dist=25, ring=56,
               name="C4 front end: synthetic 1280x720 RGB-D stream, 500 features, min_dist 25 (BASELINE.json configs[3])"),
}


def tri(k, n):
    """ping-pong index so the ring stays temporally coherent"""
    p = k % (2 * n - 2)
    return p if p < n else 2 * n - 2 - p


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons through NVML (no process is forked while a timed region runs); rank 0 only."""

    def __init__(self, gpu, period=0.05):
        super().__init__(daemon=True)
        self.gpu, self.period, self.rows, self.stop_flag, self.active = gpu, period, [], False, False
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[gpu]) if vis and vis.split(",")[gpu].isdigit() else gpu
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.h = None

    def run(self):
        nv = self.nv if self.h is not None else None
        while not self.stop_flag:
            if self.active and nv is not None:
                try:
                    self.rows.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM),
                                      nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)))
                except Exception:
                    try:
                        self.rows.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM), nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)))
                    except Exception:
                        pass
            time.sleep(self.period)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(r[0] for r in self.rows)
        bits = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        reasons = [name for b, name in bits.items() if any(r[1] & b for r in self.rows)]
        return {"sm_mhz": float(sm[len(sm) // 2]), "sm_max_mhz": float(self.max_sm), "reasons": reasons, "samples": len(self.rows),
                "source": "NVML, sampled every %d ms inside the timed regions (rank 0)" % int(self.period * 1e3)}


def pin_to_local_cpus(local_rank, n_local):
    """Give every rank a disjoint slice of the CPUs that are NUMA-local to its GPU (falls back to doing nothing)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        path = "/sys/bus/pci/devices/%s/local_cpulist" % bus.lower()[-12:]
        txt = open(path).read().strip()
        cpus = []
        for part in txt.split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        cpus = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not cpus:
            return None
        # the ranks whose GPUs share this NUMA node split its CPUs evenly
        same = [r for r in range(n_local) if _cpulist_of(r) == txt]
        k = same.index(local_rank) if local_rank in same else 0
        per = max(1, len(cpus) // max(1, len(same)))
        mine = cpus[k * per:(k + 1) * per] or cpus
        os.sched_setaffinity(0, mine)
        return "%d cpus NUMA-local to the GPU (%s)" % (len(mine), txt)
    except Exception:
        return None


def _cpulist_of(idx):
    try:
        import pynvml
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        return open("/sys/bus/pci/devices/%s/local_cpulist" % bus.lower()[-12:]).read().strip()
    except Exception:
        return None


def make_frames(seed, n, w, h):
    from ground_fusion_b200.synth import SyntheticStream
    st = SyntheticStream(seed=seed, width=w, height=h)
    gray = np.empty((n, h, w), np.uint8)
    depth = np.empty((n, h, w), np.uint16)
    for k in range(n):
        _, gray[k], depth[k] = st.frame(k)
    return gray, depth


# ---------------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline
# ---------------------------------------------------------------------------------------------------------------------
def cpu_reference(gray, depth, wl, n_steps, frames_per_step, warm_steps=1):
    """frames/s of the reference's CPU path (cv2 calls + C glue) over n_steps bounded samples; also the OpenCV-only rate."""
    import cv2
    from oracle.fe_oracle import IDC_CAM, FeatureTrackerOracleFast, PinholeCamera
    sc = wl["w"] / 640.0
    cam = PinholeCamera(IDC_CAM["fx"] * sc, IDC_CAM["fy"] * sc, IDC_CAM["cx"] * sc, IDC_CAM["cy"] * sc,
                        IDC_CAM["k1"], IDC_CAM["k2"], IDC_CAM["p1"], IDC_CAM["p2"])
    ft = FeatureTrackerOracleFast(cam, wl["max_cnt"], wl["min_dist"], 1, 1)
    n = len(gray)
    k = 0
    for _ in range(warm_steps * frames_per_step):
        ft.trackImage(k / 30.0, gray[tri(k, n)], depth[tri(k, n)]); k += 1
    ft.t_cv = 0.0
    t0 = time.perf_counter()
    for _ in range(n_steps * frames_per_step):
        ft.trackImage(k / 30.0, gray[tri(k, n)], depth[tri(k, n)]); k += 1
    dt = time.perf_counter() - t0
    done = n_steps * frames_per_step
    return {"fps": done / dt, "cv_only_fps": done / ft.t_cv, "glue_fraction": 1.0 - ft.t_cv / dt, "frames": done, "threads": cv2.getNumThreads()}


# ---------------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------------
class Ring:
    """Frames of one stream: resident in HBM and in pinned host memory."""

    def __init__(self, seed, wl, torch):
        self.n = wl["ring"]
        gray, depth = make_frames(seed, self.n, wl["w"], wl["h"])
        self.gray, self.depth = gray, depth
        self.d_gray = torch.from_numpy(gray).cuda()
        self.d_depth = torch.from_numpy(depth.view(np.int16)).cuda()
        self.h_gray = torch.from_numpy(gray).pin_memory()
        self.h_depth = torch.from_numpy(depth.view(np.int16)).pin_memory()
        fb_g, fb_d = wl["w"] * wl["h"], wl["w"] * wl["h"] * 2
        self.ptr = {"device": ([self.d_gray.data_ptr() + i * fb_g for i in range(self.n)], [self.d_depth.data_ptr() + i * fb_d for i in range(self.n)]),
                    "host": ([self.h_gray.data_ptr() + i * fb_g for i in range(self.n)], [self.h_depth.data_ptr() + i * fb_d for i in range(self.n)])}


class Stream:
    def __init__(self, ring, wl, device, offset=0):
        from ground_fusion_b200.feature_tracker import FeatureTracker
        from ground_fusion_b200.synth import idc_params8
        sc = wl["w"] / 640.0
        p8 = idc_params8()
        p8 = [p8[0] * sc, p8[1] * sc, p8[2] * sc, p8[3] * sc] + p8[4:]
        self.tr = FeatureTracker(wl["w"], wl["h"], p8, wl["max_cnt"], wl["min_dist"], 1, 1, device=device)
        self.ring, self.k, self.dev_ms, self.last_out = ring, offset, 0.0, None

    def run(self, n_steps, mode, keep_last=False):
        """n_steps batches of FRAMES_PER_STEP frames; returns the device time of the run (CUDA events on the tracker's streams).
        keep_last: the last batch also copies its results out to the caller (self.last_out, as trackBatch returns them)."""
        g, d = self.ring.ptr[mode]
        n = self.ring.n
        self.tr.timer_start()
        for s in range(n_steps):
            idx = [tri(self.k + j, n) for j in range(FRAMES_PER_STEP)]
            times = [(self.k + j) / 30.0 for j in range(FRAMES_PER_STEP)]
            want = keep_last and s == n_steps - 1
            out = self.tr.trackBatch(times, [g[i] for i in idx], [d[i] for i in idx], on_device=(mode == "device"), want=want)
            if want:
                self.last_out = out
            self.k += FRAMES_PER_STEP
        self.dev_ms = self.tr.timer_stop()
        return self.dev_ms


def run_multi(streams, n_steps, mode):
    """The same n_steps on S streams through gf_tracker_track_batch_multi: one host thread feeds all the streams."""
    from ground_fusion_b200.feature_tracker import FeatureTracker
    for s in streams:
        s.tr.timer_start()
    for _ in range(n_steps):
        times, gp, dp = [], [], []
        for s in streams:
            g, d = s.ring.ptr[mode]
            idx = [tri(s.k + j, s.ring.n) for j in range(FRAMES_PER_STEP)]
            times.append([(s.k + j) / 30.0 for j in range(FRAMES_PER_STEP)])
            gp.append([g[i] for i in idx]); dp.append([d[i] for i in idx])
            s.k += FRAMES_PER_STEP
        FeatureTracker.trackBatchMulti([s.tr for s in streams], times, gp, dp, on_device=(mode == "device"), want=False)
    for s in streams:
        s.dev_ms = s.tr.timer_stop()


def timed(streams, n_steps, mode, barrier, sampler=None, threads=False, keep_last=False):
    """K steps on every stream of this rank; wall clock between barriers.  Several streams: one host thread and
    gf_tracker_track_batch_multi, or (threads=True, for comparison) one host thread per stream."""
    assert not keep_last or len(streams) == 1
    barrier()
    if sampler is not None:
        sampler.active = True
    t0 = time.perf_counter()
    if len(streams) == 1:
        streams[0].run(n_steps, mode, keep_last)
    elif not threads:
        run_multi(streams, n_steps, mode)
    else:
        th = [threading.Thread(target=s.run, args=(n_steps, mode)) for s in streams]
        for x in th:
            x.start()
        for x in th:
            x.join()
    barrier()
    el = time.perf_counter() - t0
    if sampler is not None:
        sampler.active = False
    return el, max(s.dev_ms for s in streams)


def fe_line(wl, rings, device, n_streams, steps, warmup, barrier, sampler, reduce_max, threads=False, keep_last=False):
    """keep_last: "last_step" of the result is what the last device-resident timed step returned (see Stream.run)."""
    streams = [Stream(rings[0], wl, device, offset=17 * s) for s in range(n_streams)]
    from ground_fusion_b200 import _lib
    timed(streams, warmup, "device", barrier, threads=threads)
    l0 = _lib.lib().gf_kernel_launch_count()
    el_dev, ms_dev = timed(streams, steps, "device", barrier, sampler, threads=threads, keep_last=keep_last)
    launches = _lib.lib().gf_kernel_launch_count() - l0
    timed(streams, max(1, warmup // 2), "host", barrier, threads=threads)
    el_e2e, ms_e2e = timed(streams, steps, "host", barrier, sampler, threads=threads)
    el_dev, el_e2e, ms_dev, ms_e2e = reduce_max([el_dev, el_e2e, ms_dev, ms_e2e])
    infos = streams[0].tr.batch_infos
    for s in streams:
        s.tr.close()
    frames = n_streams * steps * FRAMES_PER_STEP
    return {"value": frames / el_dev, "e2e": frames / el_e2e, "ms_per_step": 1e3 * el_dev / steps, "ms_per_step_e2e": 1e3 * el_e2e / steps,
            "device_ms_per_step": ms_dev / steps, "device_ms_per_step_e2e": ms_e2e / steps, "streams_per_gpu": n_streams, "gpu_launches": int(launches),
            "mean_features_tracked": float(np.mean([i["n_tracked"] for i in infos])), "mean_lk_iterations": float(np.mean([i["lk_iterations"] for i in infos])),
            "last_step": streams[0].last_out}


def dump_outputs(path, batch, max_cnt):
    """One trackBatch result (per frame: observations, inlier mask, counters) as float64 arrays padded to max_cnt per frame:
    n_obs[f], obs_id[f, i] (-1 past n_obs), obs_track_cnt[f, i], obs_v[f, i, 8] (gf_obs.v: x_n y_n 1 u v vx_n vy_n depth_m),
    n_prev[f], status[f, i] (0 past n_prev), info[f, :] (gf_track_info in declaration order)."""
    from ground_fusion_b200._lib import TrackInfo
    fields = [name for name, _ in TrackInfo._fields_]
    n = len(batch)
    a = {"n_obs": np.zeros(n), "obs_id": np.full((n, max_cnt), -1.0), "obs_track_cnt": np.zeros((n, max_cnt)),
         "obs_v": np.zeros((n, max_cnt, 8)), "n_prev": np.zeros(n), "status": np.zeros((n, max_cnt)), "info": np.zeros((n, len(fields)))}
    for f, (obs, status, info) in enumerate(batch):
        m, p = len(obs), len(status)
        a["n_obs"][f], a["n_prev"][f] = m, p
        a["obs_id"][f, :m] = obs["id"]
        a["obs_track_cnt"][f, :m] = obs["track_cnt"]
        a["obs_v"][f, :m] = obs["v"]
        a["status"][f, :p] = status
        a["info"][f] = [info[k] for k in fields]
    os.makedirs(path, exist_ok=True)
    for name, arr in a.items():
        np.save(os.path.join(path, name + ".npy"), arr)


def ba_bench(device, clocks_mhz, n_windows=8, reps=200, cpu_seconds=8.0):
    """Sliding-window solves/s (C2: 11 frames, ~1.8 k visual factors, 10 IMU factors, 8 iterations max) on the GPU through
    gf_ba_solve (host descriptor in, optimised blocks out: this IS the end-to-end call) next to the CPU oracle."""
    from ground_fusion_b200 import _lib
    from ground_fusion_b200.estimator import BundleAdjuster
    from ground_fusion_b200.synth_ba import make_window
    L = _lib.lib()
    wins = [make_window(seed=100 + k)[0] for k in range(n_windows)]
    saved = [(w.para_pose.copy(), w.para_speed_bias.copy(), w.para_feature.copy(), w.para_ex_pose.copy(), w.para_td.copy()) for w in wins]
    structs = [w.struct() for w in wins]

    def restore(k):
        w, sv = wins[k], saved[k]
        w.para_pose[:] = sv[0]; w.para_speed_bias[:] = sv[1]; w.para_feature[:] = sv[2]; w.para_ex_pose[:] = sv[3]; w.para_td[:] = sv[4]
    ba = BundleAdjuster(device)
    L.gf_ba_debug_profile.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_longlong)]
    for k in range(n_windows):
        restore(k); ba.solve_struct(structs[k])
    dev_ms = 0.0; iters = 0; step_cycles = 0; step_launches = 0
    prof = (ctypes.c_longlong * 32)()
    t0 = time.perf_counter()
    for r in range(reps):
        k = r % n_windows
        restore(k)
        sm = ba.solve_struct(structs[k])
        dev_ms += sm.device_ms; iters += sm.iterations
        L.gf_ba_debug_profile(ba._h, prof)
        step_cycles += prof[30]; step_launches += prof[31]
    el = time.perf_counter() - t0
    nc, n_lm = int(sm.reduced_dim), int(sm.n_free_landmarks)
    out = {"metric": "ba_solves_per_sec", "value": reps / el, "unit": "solves/s", "ms_per_solve": 1e3 * el / reps,
           "device_ms_per_solve": dev_ms / reps, "iterations_per_solve": iters / reps,
           "workload": "C2 window: 11 frames, %d visual factors, %d IMU factors, reduced system %d + %d free landmarks, max 8 iterations"
                       % (wins[0].n_visual, wins[0].n_imu, nc, n_lm),
           "e2e": "value already includes the host->device upload of the problem and the download of the blocks"}
    # roofline of the dominant kernel (k_ba_step: tiled Cholesky on DMMA + back substitution + dogleg), per launch:
    # (nc+1)^3/3 (factorisation) + nc^2 (two triangular solves) + 3 n_lm nc (landmark back substitution, dogleg terms) FMA
    dfma, dmma = ctypes.c_double(0), ctypes.c_double(0)
    L.gf_probe_fp64.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
    L.gf_probe_fp64(device, ctypes.byref(dfma), ctypes.byref(dmma))
    fma = (nc + 1) ** 3 / 3.0 + nc * nc + 3.0 * n_lm * nc
    mhz = clocks_mhz or 1965.0
    t_launch = (step_cycles / max(1, step_launches)) / (mhz * 1e6)
    ach = 2.0 * fma / t_launch / 1e9 if t_launch > 0 else None
    n_sm = 148
    out["roofline"] = {"kernel": "k_ba_step (one CTA: 8x8-tile left-looking Cholesky on DMMA.8x8x4, back substitution, dogleg, candidate)",
                       "bound": "tensor", "unit": "GFLOP/s (FP64)", "achieved": ach, "peak": dmma.value, "frac": ach / dmma.value if ach else None,
                       "peak_source": "gf_probe_fp64: DMMA.8x8x4 on all SMs, measured in this run (plain DFMA: %.0f GFLOP/s)" % dfma.value,
                       "frac_of_one_sm": ach / (dmma.value / n_sm) if ach else None,
                       "algorithmic_flops_per_launch": 2.0 * fma, "launch_us": 1e6 * t_launch, "launches_per_solve": step_launches / reps,
                       "time_share_of_solve": (step_cycles / (mhz * 1e3)) / dev_ms if dev_ms else None, "traffic": None,
                       "note": "a single window is a dependent chain of %d panel factorisations on ONE SM (latency-bound: rsqrt chain of the 8x8 diagonal "
                               "tiles); the kernel cannot use more than 1/%d of the device, see frac_of_one_sm" % ((nc + 8) // 8, n_sm)}
    # the marginalisation that ends Estimator::optimization() on a keyframe (MARGIN_OLD), on the solved window
    restore(0); ba.solve_struct(structs[0])
    ba.marginalize_old(wins[0])
    mms = []
    for _ in range(5):
        ba.marginalize_old(wins[0]); mms.append(ba.last_marg_ms)
    out["marginalize_old"] = {"device_ms": float(np.median(mms)), "note": "gf_ba_marginalize_old on the solved C2 window"}
    ba.close()
    # independent windows (several estimators sharing one GPU): one gf_ba handle and one host thread per stream
    n_str = 4
    sets = []
    for t in range(n_str):
        ws = [make_window(seed=200 + 10 * t + k)[0] for k in range(2)]
        sets.append((ws, [w.struct() for w in ws], [(w.para_pose.copy(), w.para_speed_bias.copy(), w.para_feature.copy()) for w in ws], BundleAdjuster(device)))

    def worker(t, n):
        ws, st, sv, b = sets[t]
        for r in range(n):
            k = r % len(ws)
            ws[k].para_pose[:] = sv[k][0]; ws[k].para_speed_bias[:] = sv[k][1]; ws[k].para_feature[:] = sv[k][2]
            b.solve_struct(st[k])
    for t in range(n_str):
        worker(t, 2)
    th = [threading.Thread(target=worker, args=(t, reps)) for t in range(n_str)]
    t0 = time.perf_counter()
    for x in th:
        x.start()
    for x in th:
        x.join()
    elc = time.perf_counter() - t0
    out["concurrent_streams"] = {"streams": n_str, "value": n_str * reps / elc, "unit": "solves/s",
                                 "note": "aggregate of %d independent windows solved concurrently on one GPU (one gf_ba handle + host thread each)" % n_str}
    for s_ in sets:
        s_[3].close()
    from oracle import ba_oracle
    t0 = time.perf_counter(); done = 0
    while time.perf_counter() - t0 < cpu_seconds:
        k = done % n_windows
        restore(k); ba_oracle.solve(wins[k]); done += 1
    dt = time.perf_counter() - t0
    out["cpu_baseline"] = {"value": done / dt, "unit": "solves/s", "cores": 1, "kind": "port",
                           "sample": "%d solves of the same windows, oracle/ba_oracle.c (block-sparse Schur, gcc -O3 as the reference, 1 thread)" % done}
    out["speedup_vs_cpu"] = out["value"] / out["cpu_baseline"]["value"]
    restore(0); ba_oracle.solve(wins[0])
    t0 = time.perf_counter(); ba_oracle.marginalize_old(wins[0])
    out["marginalize_old"]["cpu_oracle_ms"] = 1e3 * (time.perf_counter() - t0)
    return out


def ate_replay(device, n_frames=64):
    """BASELINE.json's accuracy bar: the same synthetic RGB-D + IMU sequence replayed through the whole loop (front end ->
    FeatureManager -> optimization() -> marginalisation -> slideWindow, ground_fusion_b200/replay.py) once on the GPU library
    and once on the CPU oracles; ATE of each against the stream's ground truth and the largest distance between the two
    estimated trajectories.  The bar is |ATE_gpu - ATE_cpu| <= 1 mm."""
    import numpy as np
    from ground_fusion_b200.estimator import BundleAdjuster
    from ground_fusion_b200.feature_manager import FeatureManager
    from ground_fusion_b200.feature_tracker import FeatureTracker
    from ground_fusion_b200.replay import replay
    from ground_fusion_b200.synth import IDC_CAM, SyntheticStream
    from oracle.replay_adapters import oracle_components
    cam = dict(IDC_CAM, k1=0.0, k2=0.0, p1=0.0, p2=0.0)       # the renderer is an ideal pinhole
    p8 = [cam[k] for k in ("fx", "fy", "cx", "cy", "k1", "k2", "p1", "p2")]
    tr, fm, ba = oracle_components(cam, depth_threshold=4.0)
    t0 = time.perf_counter()
    want = replay(SyntheticStream(seed=0), tr, fm, ba, n_frames)
    t_cpu = time.perf_counter() - t0
    gtr, gfm, gba = FeatureTracker(640, 480, p8, 150, 30, 1, 1, device=device), FeatureManager(depth_threshold=4.0, device=device), BundleAdjuster(device)
    t0 = time.perf_counter()
    got = replay(SyntheticStream(seed=0), gtr, gfm, gba, n_frames)
    t_gpu = time.perf_counter() - t0
    gtr.close(); gba.close()
    diff = float(np.linalg.norm(got["P_est"] - want["P_est"], axis=1).max())
    return {"frames": n_frames, "ate_gpu_m": got["ate_m"], "ate_cpu_oracle_m": want["ate_m"], "abs_ate_difference_m": abs(got["ate_m"] - want["ate_m"]),
            "max_trajectory_difference_m": diff, "within_1mm": bool(abs(got["ate_m"] - want["ate_m"]) <= 1e-3),
            "solves": len(got["iterations"]), "margin_old": got["n_margin_old"], "margin_second_new": got["n_margin_second_new"],
            "same_iteration_counts": bool(list(got["iterations"]) == list(want["iterations"])),
            "wall_s": {"gpu_pipeline_incl_rendering": t_gpu, "cpu_oracle_pipeline_incl_rendering": t_cpu},
            "note": "synthetic 640x480 RGB-D + IMU stream (seed 0), first 11 frames initialised from ground truth (the reference's SfM initialisation is outside the path), depth_threshold 4 m"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-seconds", type=float, default=8.0)
    ap.add_argument("--no-extras", action="store_true", help="only the headline C2 line (no stream sweep, C3/C4, BA)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step of the headline run returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.steps < 1):
        ap.error("--dump-outputs needs --impl ours and at least one timed step")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    wl = WORKLOADS["C2"]
    cfg = {"workload": wl["name"], "frames_per_step": FRAMES_PER_STEP, "frames_ring": wl["ring"],
           "l2_policy": "inputs larger than L2 (ring of %d distinct frames = %.0f MB per stream)" % (wl["ring"], wl["ring"] * wl["w"] * wl["h"] * 3 / 1e6),
           "streams_per_gpu": 1, "parallelism": "one independent stream per GPU"}

    if args.impl == "reference":
        if rank != 0:
            return
        gray, depth = make_frames(0, 60, wl["w"], wl["h"])
        fps_step = 20                     # each step = a bounded sample (20 frames) of the 100-frame batch
        r = cpu_reference(gray, depth, wl, max(1, args.steps), fps_step, warm_steps=max(1, min(args.warmup, 3)))
        v = r["fps"]
        print(json.dumps({"impl": "reference", "metric": "tracker_frames_per_sec", "value": v, "unit": "frames/s", "n_gpus": args.gpus,
                          "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * fps_step / v, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "u8/f32 (OpenCV)", "data": "synthetic", "config": cfg,
                          "cpu_baseline": {"value": v, "unit": "frames/s", "cores": r["threads"], "kind": "port",
                                           "sample": "%d frames of the C2 stream per step (bounded sample of the 100-frame batch), %d steps; cv2 %d threads" % (fps_step, args.steps, r["threads"]),
                                           "opencv_calls_only": r["cv_only_fps"], "glue_fraction": r["glue_fraction"]},
                          "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    # libraries (NCCL's version banner, torchrun warnings) may write to fd 1: keep it for the one JSON line, send the rest to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(json_fd, (json.dumps(obj) + "\n").encode())

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    affinity = pin_to_local_cpus(local, int(os.environ.get("LOCAL_WORLD_SIZE", str(world))))
    from ground_fusion_b200 import _lib

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(vals):
        if dist is None:
            return vals
        t = torch.tensor(vals, device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]

    sampler = None
    if rank == 0:
        sampler = ClockSampler(local); sampler.start()
    ring = Ring(rank, wl, torch)
    head = fe_line(wl, [ring], local, 1, args.steps, args.warmup, barrier, sampler, reduce_max, keep_last=bool(args.dump_outputs))
    clocks = sampler.summary() if sampler is not None else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, head["last_step"], wl["max_cnt"])

    extra = {}
    if world > 1 and not args.no_extras:
        # C5: 300 features per stream, one stream per GPU
        w5 = WORKLOADS["C3"]
        ring5 = Ring(rank, w5, torch)
        c5 = fe_line(w5, [ring5], local, 1, args.steps, args.warmup, barrier, None, reduce_max)
        extra["C5"] = {"workload": w5["name"] + ", one stream per GPU", "value": world * c5["value"], "e2e": world * c5["e2e"], "unit": "frames/s",
                       "ms_per_step": c5["ms_per_step"]}
        del ring5
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm = peaks.get("hbm_gbs", 6650.0)
    out = {"metric": "tracker_frames_per_sec", "value": world * head["value"], "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "u8/i32 fixed point + f32 (LK, min-eig), f64 (box sums, undistortion)", "data": "synthetic", "config": cfg,
           "device_ms_per_step": head["device_ms_per_step"], "device_ms_per_step_e2e": head["device_ms_per_step_e2e"],
           "timing": "value/e2e: wall clock between barrier+synchronize around K steps of %d frames, max over ranks; device_ms_per_step*: CUDA events "
                     "around the same frames on the tracker's streams (first copy .. last result copy), max over ranks" % FRAMES_PER_STEP,
           "frames_in_flight": 2, "mean_features_tracked": head["mean_features_tracked"],
           "e2e": {"value": world * head["e2e"], "unit": "frames/s", "h2d_bytes_per_step": FRAMES_PER_STEP * wl["w"] * wl["h"] * 3,
                   "d2h_bytes_per_step": FRAMES_PER_STEP * (wl["max_cnt"] * 72 + 40 + 1024), "ms_per_step": head["ms_per_step_e2e"]},
           "gpu_launches": head["gpu_launches"], "gpu_launches_note": "kernels launched by libgf_b200 (rank 0) inside the K timed device-resident steps",
           "clocks": clocks, "cpu_affinity": affinity}
    out.update(extra)

    # ---- stage breakdown + roofline of the dominant kernel (profiling mode: one frame at a time, event records only); rank 0, any N ----
    try:
        from ground_fusion_b200.feature_tracker import FeatureTracker
        from ground_fusion_b200.synth import idc_params8
        tr = FeatureTracker(wl["w"], wl["h"], idc_params8(), wl["max_cnt"], wl["min_dist"], 1, 1, device=local)
        g, d = ring.ptr["device"]
        for k in range(30):
            tr.trackDevice(k / 30.0, g[tri(k, ring.n)], d[tri(k, ring.n)])
        tr.set_profiling(True)
        stage = {}; iters = 0; nprev = 0
        for k in range(30, 80):
            tr.trackDevice(k / 30.0, g[tri(k, ring.n)], d[tri(k, ring.n)])
            for s, v in tr.last_stage_ms().items():
                stage[s] = stage.get(s, 0.0) + v / 50.0
            iters += tr.last_info["lk_iterations"] / 50.0; nprev += tr.last_info["n_prev"] / 50.0
        tr.set_profiling(False); tr.close()
        lk_bytes = nprev * 6 * 23 * 23 + iters * 22 * 22        # SURVEY 8d: window gathers (4 fwd + 2 bwd levels) + one 22x22 window per LK iteration
        lk_s = stage.get("lk", 0.0) / 1e3
        out["stage_ms"] = stage
        out["roofline"] = {"kernel": "k_track (fwd 4-level + reverse 2-level LK, one 8-warp CTA per feature)", "bound": "hbm",
                           "achieved": (lk_bytes / lk_s / 1e9) if lk_s > 0 else None, "peak": hbm, "unit": "GB/s",
                           "frac": (lk_bytes / lk_s / 1e9 / hbm) if lk_s > 0 else None,
                           "traffic": 899072, "traffic_source": "dram__bytes_read+write of one k_track launch, profiles/r2_ncu_k_track_full.txt",
                           "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                           "algorithmic_bytes_per_launch": lk_bytes, "kernel_ms": stage.get("lk"),
                           "note": "latency-bound by construction: per feature a chain of ~22 dependent LK iterations, each 105 dependent FADDs in OpenCV lane order; "
                                   "throughput comes from concurrent streams (see streams)"}
    except Exception as e_:      # the headline line must survive
        out["roofline"] = {"error": repr(e_)}
    if world == 1 and not args.no_extras:
        # ---- several independent streams on one GPU ----
        sweep = {}
        for ns in (2, 4, 8, 16):
            r = fe_line(wl, [ring], local, ns, max(4, args.steps // 2), 2, barrier, None, reduce_max)
            sweep[str(ns)] = {"value": r["value"], "e2e": r["e2e"]}
        sweep["1"] = {"value": head["value"], "e2e": head["e2e"]}
        r = fe_line(wl, [ring], local, 8, max(4, args.steps // 2), 2, barrier, None, reduce_max, threads=True)
        out["streams"] = {"unit": "frames/s", "per_streams_per_gpu": sweep,
                          "eight_streams_one_host_thread_each": {"value": r["value"], "e2e": r["e2e"]},
                          "note": "independent trackers (gf_tracker handles) sharing one B200, all fed by ONE host thread through gf_tracker_track_batch_multi; eight_streams_one_host_thread_each = the same 8 trackers driven by 8 host threads calling gf_tracker_track_batch; e2e saturates on the host link (0.92 MB per frame: 31 k frames/s = 28.5 GB/s); C2 workload"}
        # ---- the other configurations ----
        cfgs = {}
        for name in ("C3", "C4"):
            w2 = WORKLOADS[name]
            ring2 = ring if (w2["w"], w2["h"]) == (wl["w"], wl["h"]) else Ring(0, w2, torch)
            r = fe_line(w2, [ring2], local, 1, max(4, args.steps // 2), 2, barrier, None, reduce_max)
            cpu = cpu_reference(ring2.gray[:40], ring2.depth[:40], w2, 1, 40 if name == "C3" else 20)
            cfgs[name] = {"workload": w2["name"], "value": r["value"], "e2e": r["e2e"], "unit": "frames/s", "ms_per_step": r["ms_per_step"],
                          "mean_features_tracked": r["mean_features_tracked"],
                          "cpu_baseline": {"value": cpu["fps"], "opencv_calls_only": cpu["cv_only_fps"], "cores": cpu["threads"], "kind": "port", "sample": "%d frames" % cpu["frames"]}}
            if ring2 is not ring:
                del ring2
        out["configs"] = cfgs
        # ---- CPU baseline of the headline workload ----
        cpu = cpu_reference(ring.gray[:60], ring.depth[:60], wl, max(1, int(args.cpu_seconds / 0.6)), 100, warm_steps=1)
        out["cpu_baseline"] = {"value": cpu["fps"], "unit": "frames/s", "cores": cpu["threads"], "kind": "port",
                               "sample": "%d frames of the same C2 stream: the reference's three OpenCV calls (cv2 4.13) + its glue in C (FeatureTrackerOracleFast)" % cpu["frames"],
                               "opencv_calls_only": cpu["cv_only_fps"], "glue_fraction": cpu["glue_fraction"]}
        try:
            out["ba"] = ba_bench(local, (clocks or {}).get("sm_mhz"), cpu_seconds=min(args.cpu_seconds, 8.0))
        except Exception as e:      # the FE line must survive a BA problem
            out["ba"] = {"error": repr(e)}
        try:
            out["ate"] = ate_replay(local)
        except Exception as e:
            out["ate"] = {"error": repr(e)}
    if sampler is not None:
        sampler.stop_flag = True
    emit(out)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
