#!/usr/bin/env python
"""bench.py -- stereo frames/s of the HybVIO hot path (pyramid + LK + EKF) on B200, BASELINE.json's metric.

  python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (CUDA, libhybvio_b200.so)
  python bench.py --impl reference ...                            the reference's own CPU path (oracle/_ref)
  python bench.py ... --dump-outputs DIR                          also writes what the last timed step computed to DIR/*.npy

A "step" is ONE stereo frame of BASELINE config 2 (EuRoC V1_02-shaped: 752x480 stereo, 150 features, 4-level pyramid,
31x31 window, EKF state dimension 160) pushed through the whole hot path of one VIO session:
    2 pyramids (one launch) -> LK prev-left -> left with predicted initial flow -> LK left -> right
    -> 10 x (EKF predict + normalizeQuaternions(true)) (200 Hz IMU at 20 fps; backend.cpp:734-735) -> 20 visual-track outlier checks, the 5 designated ones followed by
       their update (n = 8/20/40/84 rows, SURVEY.md 8(d)) -> maintainPositiveSemiDefinite -> pose augmentation.
Frames of one session are strictly sequential, so one stream per GPU is a latency-bound workload; --gpus N runs N
independent sessions, one per GPU (BASELINE config 3; no data-path collective, NCCL only for the start barrier and
the max-over-ranks reduction of the device time).

`value`  = frames/s with every input already resident in HBM, no host synchronisation inside the timed region.
`e2e`    = the same frames through the host-buffer C ABI the reference-side adapters call: each step copies its two
           frames host->device from pinned memory, every LK call and every outlier check returns its result to the host
           (the reference interface is synchronous there: src/odometry/backend.cpp:1158-1161), and the pose is read back.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

T_PROCESS_START = time.monotonic()
# Report-only extras (child processes, after the headline measurement): none is started later than EXTRAS_START_BY seconds into the
# run and none gets more than EXTRAS_TIMEOUT seconds, so that the default `python bench.py` stays within a few minutes even if an
# extra hangs (they exercise opt-in kernels). HV_BENCH_NO_EXTRAS=1 switches them off.
EXTRAS_START_BY = 180.0
EXTRAS_TIMEOUT = 120.0

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

W, H, NFEAT, WIN, MAXLEVEL, TRAIL = 752, 480, 150, 31, 3, 20
STEREO = True
CONFIG_ID = 2
VISUAL_R = 0.05
FOCAL = 458.0
# e2e_adapter: the outlier check and the update use DIFFERENT noise levels, 30 : 1 like odometry.trackChiTestOutlierR (1.5) : odometry.visualR
# (0.05) (backend.cpp:995-997); the check keeps the noise level the synthetic measurements were generated for
CHI_OUTLIER_R, UPDATE_R = VISUAL_R, VISUAL_R / 30.0
N_ROWS = (8, 20, 40, 84)            # rows of the visual measurement models, cycled (SURVEY.md 8(d))
CHECKS, UPDATES, PREDICTS = 20, 5, 10
# BASELINE.json configs that fit one GPU. 2 is the headline (the metric is quoted on it); 4 and 1 via --config.
CONFIGS = {
    2: dict(W=752, H=480, NFEAT=150, MAXLEVEL=3, TRAIL=20, STEREO=True, N_ROWS=(8, 20, 40, 84),
            name="BASELINE config 2: EuRoC V1_02-shaped stereo 752x480, 150 features, 4-level pyramid, win 31, EKF N=160 (trail 20)"),
    4: dict(W=512, H=512, NFEAT=200, MAXLEVEL=3, TRAIL=6, STEREO=True, N_ROWS=(8, 12, 20, 28),
            name="BASELINE config 4: TUM-VI-shaped stereo 512x512, 200 features, 4-level pyramid, win 31, EKF N=62 (trail 6)"),
    1: dict(W=752, H=480, NFEAT=100, MAXLEVEL=2, TRAIL=20, STEREO=False, N_ROWS=(4, 10, 20, 42),
            name="BASELINE config 1: EuRoC MH_01-shaped mono 752x480, 100 features, 3-level pyramid, win 31, EKF N=160 (trail 20)"),
}
CONFIG_NAME = CONFIGS[2]["name"]
IMU_OPS = 2 * PREDICTS               # every predict is followed by normalizeQuaternions(true) (src/odometry/backend.cpp:734-735)
POOL_FRAMES = int(os.environ.get("HV_BENCH_POOL_FRAMES", "128"))   # stereo pairs in the frame pool: 128 * 2 * 361 KB = 92 MB
POOL_EKF = 64                       # frames of EKF inputs: 64 * 736 KB = 47 MB  (together 139 MB > 126 MB of L2)
PYR_BYTES = 2_397_000               # algorithmic bytes per image (SURVEY.md 8(d))
LK_BYTES = NFEAT * 4 * 6144 + 12 * NFEAT
NCAM = 2


def set_config(cid):
    """Rebinds the workload constants to a BASELINE config (before any session exists)."""
    global W, H, NFEAT, MAXLEVEL, TRAIL, STEREO, N_ROWS, CONFIG_ID, CONFIG_NAME, PYR_BYTES, LK_BYTES, NCAM
    c = CONFIGS[cid]
    W, H, NFEAT, MAXLEVEL, TRAIL, STEREO, N_ROWS = c["W"], c["H"], c["NFEAT"], c["MAXLEVEL"], c["TRAIL"], c["STEREO"], c["N_ROWS"]
    CONFIG_ID, CONFIG_NAME, NCAM = cid, c["name"], 2 if c["STEREO"] else 1
    sizes = [(W, H)]
    for _ in range(MAXLEVEL):
        sizes.append(((sizes[-1][0] + 1) // 2, (sizes[-1][1] + 1) // 2))
    px = [a * b for a, b in sizes]
    PYR_BYTES = px[0] + sum(px[1:]) + 4 * sum(px)            # read level 0, write gray 1..L, write (Ix, Iy) int16 of every level (SURVEY.md 8(d))
    LK_BYTES = NFEAT * (MAXLEVEL + 1) * 6144 + 12 * NFEAT


def METRIC():
    return "stereo frames/sec (752x480, 150 tracks)" if CONFIG_ID == 2 else f"{'stereo' if STEREO else 'mono'} frames/sec ({W}x{H}, {NFEAT} tracks)"


def frame_index(k):                 # ping-pong through the pool so that consecutive steps are consecutive frames
    p = 2 * (POOL_FRAMES - 1)
    j = k % p
    return j if j < POOL_FRAMES else p - j


def ekf_rows(c):
    n = N_ROWS[c % len(N_ROWS)]
    return n, min(20 + 7 * TRAIL, 20 + 7 * max(1, n // (2 * NCAM)))     # 2 rows per pose and camera; H truncated to the last used pose


class Inputs:
    """Deterministic synthetic inputs of one session (SURVEY.md 8(d)), generated with torch on `device`."""

    def __init__(self, device, seed=0):
        import torch
        from hybvio_b200 import synth
        self.torch = torch
        self.frames = synth.stereo_frames_torch(0, POOL_FRAMES, W, H, seed=42 + seed, device=device)    # (P, 2, H, W) u8
        self.points = synth.interior_points(NFEAT, W, H, seed=7 + seed)
        rng = np.random.RandomState(3 + seed)
        # predicted initial flow = true flow of the synthetic stream + <= 1 px error (tracker.cpp:59-63 predictor)
        self.init_noise = rng.uniform(-1, 1, (POOL_FRAMES, NFEAT, 2)).astype(np.float32)
        self.flow = np.array([synth.true_flow(j, j + 1) for j in range(POOL_FRAMES)], np.float32)
        irng = np.random.RandomState(11 + seed)
        self.imu = np.zeros((POOL_EKF * PREDICTS, 6))
        for i in range(len(self.imu)):
            self.imu[i, :3] = np.array([0, 0, 0.2]) + irng.normal(0, 0.05, 3)
            self.imu[i, 3:] = np.array([0.3 * np.sin(0.01 * i), 0.2 * np.cos(0.013 * i), 9.819]) + irng.normal(0, 0.2, 3)
        # EKF measurement pool: per frame CHECKS x (H n x l column-major, f, y) packed in one fp64 buffer
        self.ekf_off = []
        off = 0
        for c in range(CHECKS):
            n, l = ekf_rows(c)
            self.ekf_off.append((off, n, l))
            off += n * l + 2 * n
        self.ekf_stride = off
        pool = np.zeros((POOL_EKF, off))
        for fr in range(POOL_EKF):
            for c, (o, n, l) in enumerate(self.ekf_off):
                pool[fr, o:o + n * l] = rng.normal(0, 0.1, n * l)
                f = rng.normal(0, 0.5, n)
                # designated update slots (c < UPDATES) and most others are consistent measurements; every fourth is gross
                y = f + rng.normal(0, 0.02 if (c < UPDATES or c % 4) else 40.0, n)
                pool[fr, o + n * l:o + n * l + n] = f
                pool[fr, o + n * l + n:o + n * l + 2 * n] = y
        self.ekf_pool = pool

    def init_guess(self, jp, j):
        d = self.flow[min(jp, j)] * (1.0 if j > jp else -1.0)
        return (self.points + d + self.init_noise[j]).astype(np.float32)


# ------------------------------------------------------------------------------------------------ our arm
class Session:
    """One VIO session on one GPU: Tracker-side pyramids + LK and the EKF, all on one CUDA stream."""

    def __init__(self, device_index, inputs):
        import torch
        from hybvio_b200 import capi
        self.torch, self.capi, self.inp = torch, capi, inputs
        self.dev = torch.device("cuda", device_index)
        # two CUDA streams per session: A = tracker (pyramids, LK), B = EKF. Real data dependencies are kept with events:
        # LK(k) waits for the EKF result of frame k-1 (the flow predictor reads the EKF poses, src/tracker/tracker.cpp:59-63),
        # the visual updates of frame k wait for LK(k); pyramid(k+1) and predict(k+1) overlap with what they do not depend on.
        self.stream = torch.cuda.Stream(self.dev)
        self.stream_b = torch.cuda.Stream(self.dev)
        self.ctx = capi.Context(device_index, stream=self.stream.cuda_stream)
        self.ctx_b = capi.Context(device_index, stream=self.stream_b.cuda_stream)
        self.pyr = [self.ctx.pyramid(W, H, WIN, MAXLEVEL) for _ in range(4)]     # prevL, prevR, curL, curR
        p = capi.EkfParams()
        capi.load().hv_ekf_default_params(__import__("ctypes").byref(p))
        p.camera_trail_length = TRAIL
        self.ekf = capi.Ekf(self.ctx_b, p)
        self.ev_ekf = torch.cuda.Event()
        self.ev_lk = torch.cuda.Event()
        self.overlap = os.environ.get("HV_BENCH_NO_OVERLAP") is None
        with torch.cuda.stream(self.stream):
            self.d_frames = inputs.frames.to(self.dev)
            self.d_points = torch.from_numpy(inputs.points).to(self.dev)
            self.d_init = torch.from_numpy(np.stack([np.stack([inputs.init_guess(j - 1, j) for j in range(1, POOL_FRAMES)]),
                                                     np.stack([inputs.init_guess(j + 1, j) for j in range(0, POOL_FRAMES - 1)])])).to(self.dev)
            self.d_next = torch.zeros((NFEAT, 2), dtype=torch.float32, device=self.dev)
            self.d_next2 = torch.zeros((NFEAT, 2), dtype=torch.float32, device=self.dev)
            self.d_status = torch.zeros(NFEAT, dtype=torch.uint8, device=self.dev)
            self.d_ts = torch.zeros(NFEAT, dtype=torch.int32, device=self.dev)
            self.d_ekf_pool = torch.from_numpy(inputs.ekf_pool).to(self.dev)
            self.d_res = torch.zeros(2, dtype=torch.float64, device=self.dev)
            self.d_mean = torch.zeros(20, dtype=torch.float64, device=self.dev)
        # host copy of the measurement pool in page-locked memory (the e2e contract: inputs come from pinned host memory)
        self.h_ekf_pool = torch.from_numpy(inputs.ekf_pool).pin_memory()
        # per-frame EKF op lists (hv_ekf_run_*: one crossing of the language boundary per frame)
        self.ops_dev, self.ops_host = [], []
        nops = IMU_OPS + CHECKS + 2
        for fr in range(POOL_EKF):
            od, oh = (capi.EkfOp * nops)(), (capi.EkfOp * nops)()
            for ops, base in ((od, self.d_ekf_pool[fr].data_ptr()), (oh, self.h_ekf_pool[fr].data_ptr())):
                for s_ in range(PREDICTS):
                    u = inputs.imu[fr * PREDICTS + s_]
                    ops[2 * s_].kind = capi.OP_PREDICT
                    for q in range(3):
                        ops[2 * s_].gyro[q] = u[q]; ops[2 * s_].acc[q] = u[3 + q]
                    ops[2 * s_ + 1].kind, ops[2 * s_ + 1].index = capi.OP_NORMALIZE, 1     # normalizeQuaternions(true)
                for c, (o, n, l) in enumerate(inputs.ekf_off):
                    op = ops[IMU_OPS + c]
                    op.kind, op.n, op.l, op.mode, op.r, op.rmse_thr = capi.OP_VISUAL, n, l, (2 if c < UPDATES else 0), VISUAL_R, -1.0
                    op.H, op.f, op.y = base + 8 * o, base + 8 * (o + n * l), base + 8 * (o + n * l + n)
                ops[IMU_OPS + CHECKS].kind = capi.OP_SYMMETRIZE
                ops[IMU_OPS + CHECKS + 1].kind = capi.OP_AUGMENT
                ops[IMU_OPS + CHECKS + 1].index = -1
            self.ops_dev.append(od); self.ops_host.append(oh)
        self.nops = nops
        self.h_frames = inputs.frames.cpu().pin_memory()
        self.h_pose = torch.zeros(self.ekf.N, dtype=torch.float64).pin_memory()
        self.t = 0.0
        self.k = 0
        self.prev_j = 0
        self.ekf.initialize_orientation(inputs.imu[0, 3:])
        # prime "previous frame" pyramids
        self.ctx.build_pyramids(self.pyr[0:NCAM], [self.d_frames[0, c] for c in range(NCAM)], device=True)
        self.ctx.sync(); self.ctx_b.sync()
        torch.cuda.synchronize()
        self.ev_ekf.record(self.stream_b)

    def _ekf_inputs(self, k):
        return k % POOL_EKF

    def step_device(self):
        """One frame, everything resident in HBM, no host synchronisation."""
        self.k += 1
        j = frame_index(self.k)
        ctx, inp, A, B = self.ctx, self.inp, self.stream, self.stream_b
        cur = self.pyr[2:4]
        ctx.build_pyramids(cur[:NCAM], [self.d_frames[j, c] for c in range(NCAM)], device=True)    # A, no dependency
        fr = self._ekf_inputs(self.k)
        ops = self.ops_dev[fr]
        for s in range(PREDICTS):
            self.t += 0.005
            ops[2 * s].t = self.t
        if not self.overlap:
            A.wait_stream(B); B.wait_stream(A)
        self.ekf.run_device(ops, IMU_OPS)                                                          # B: IMU burst (queued) ...
        self.ekf.predicted_mean_device(self.d_mean.data_ptr())                                     # ... its mean part first: all the flow predictor reads
        self.ev_ekf.record(B)
        self.ekf.flush()                                                                           # ... then the full launch, beside the tracker
        A.wait_event(self.ev_ekf)                                                                  # the flow predictor reads the pose propagated to this frame
        init = self.d_init[0, j - 1] if j > self.prev_j else self.d_init[1, j]
        with self.torch.cuda.stream(A):
            self.d_next.copy_(init)                               # predicted flow (host callback in the reference)
        ctx.lk_track_device(self.pyr[0], cur[0], self.d_points, self.d_next, self.d_status, self.d_ts, NFEAT, True)
        if STEREO:
            ctx.lk_track_device(cur[0], cur[1], self.d_next, self.d_next2, self.d_status, self.d_ts, NFEAT, False)
        self.ev_lk.record(A)
        B.wait_event(self.ev_lk)                                                                   # visual updates need the tracks
        self.ekf.run_device(ctypes_slice(ops, IMU_OPS, self.nops - IMU_OPS), self.nops - IMU_OPS)
        self.pyr = self.pyr[2:4] + self.pyr[0:2]
        self.prev_j = j

    def step_e2e(self):
        """The same frame through the host-buffer C ABI (what the reference-side adapters call)."""
        self.k += 1
        j = frame_index(self.k)
        ctx, inp = self.ctx, self.inp
        cur = self.pyr[2:4]
        ctx.build_pyramids(cur[:NCAM], [self.h_frames[j, c] for c in range(NCAM)], device=False)     # H2D inside
        init = inp.init_guess(self.prev_j, j)
        nxt, st, ts = ctx.lk_track(self.pyr[0], cur[0], inp.points, init)                           # H2D + D2H + sync
        if STEREO:
            nxt2, st2, ts2 = ctx.lk_track(cur[0], cur[1], nxt)
        fr = self._ekf_inputs(self.k)
        ops = self.ops_host[fr]
        for s in range(PREDICTS):
            self.t += 0.005
            ops[2 * s].t = self.t
        # 20 synchronous round trips (every check returns its VuOutlierStatus to the host) + state read-back
        st, chi2, m = self.ekf.run_host(ops, self.nops, want_m=True)
        self.pyr = self.pyr[2:4] + self.pyr[0:2]
        self.prev_j = j
        return m

    def run_e2e_native(self, nframes):
        """`nframes` consecutive frames through hybvio_b200/libhv_e2e_driver.so (native caller of the host-buffer C ABI:
        same calls as step_e2e, without the Python interpreter in the timed region). Returns device milliseconds."""
        import ctypes
        capi = self.capi
        drv = ctypes.CDLL(os.path.join(ROOT, "hybvio_b200", "libhv_e2e_driver.so"))

        class Frame(ctypes.Structure):
            _fields_ = [("left", ctypes.c_void_p), ("right", ctypes.c_void_p), ("stride", ctypes.c_size_t), ("init_xy", ctypes.c_void_p),
                        ("ops", ctypes.POINTER(capi.EkfOp)), ("nops", ctypes.c_int)]
        frames = (Frame * nframes)()
        keep = []
        for i in range(nframes):
            self.k += 1
            j = frame_index(self.k)
            init = np.ascontiguousarray(self.inp.init_guess(self.prev_j, j))
            src = self.ops_host[self._ekf_inputs(self.k)]
            ops = (capi.EkfOp * self.nops)()
            ctypes.memmove(ops, src, ctypes.sizeof(ops))
            for s_ in range(PREDICTS):
                self.t += 0.005
                ops[2 * s_].t = self.t
            keep += [init, ops]
            fr = frames[i]
            fr.left, fr.right, fr.stride = self.h_frames[j, 0].data_ptr(), (self.h_frames[j, 1].data_ptr() if STEREO else None), W
            fr.init_xy, fr.ops, fr.nops = init.ctypes.data, ops, self.nops
            self.prev_j = j
        P = (ctypes.c_void_p * 4)(*[p.h for p in self.pyr])
        pose = (ctypes.c_double * 20)()
        ms = ctypes.c_float(0.0)
        phases = (ctypes.c_double * 4)()
        drv.hv_e2e_run_phases.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                          ctypes.POINTER(Frame), ctypes.c_int, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_float),
                                          ctypes.POINTER(ctypes.c_double)]
        capi.check(drv.hv_e2e_run_phases(self.ctx.h, self.ctx_b.h, P, self.ekf.h, self.inp.points.ctypes.data, NFEAT, frames, nframes, pose,
                                         ctypes.byref(ms), phases), "hv_e2e_run")
        self.e2e_host_phase_us = {k: round(phases[i] / nframes, 2) for i, k in enumerate(("pyramids_submit", "lk_temporal", "lk_stereo", "ekf_ops"))}
        ht = (ctypes.c_double * 4)()
        if capi.load().hv_ekf_debug_host_times(self.ekf.h, ht) == 0:      # the LAST frame's measurement list: issue / wait split of its host time
            self.e2e_host_phase_us["ekf_list_last_frame"] = {"issue_us": round(ht[0], 1), "wait_us": round(ht[1], 1), "total_us": round(ht[2], 1), "ops": int(ht[3])}
        by_handle = {p.h.value: p for p in self.pyr}
        self.pyr = [by_handle[P[i]] for i in range(4)]
        return float(ms.value), np.array(pose)

    def run_dev_native(self, nframes):
        """`nframes` consecutive frames of the device-resident loop through hybvio_b200/libhv_e2e_driver.so (hv_dev_run: the
        calls of step_device issued by a native caller, so that the launch rate does not depend on the Python interpreter).
        Returns device milliseconds (CUDA events on the tracker stream around the whole loop, both streams drained)."""
        import ctypes
        capi = self.capi
        drv = ctypes.CDLL(os.path.join(ROOT, "hybvio_b200", "libhv_e2e_driver.so"))

        class DevFrame(ctypes.Structure):
            _fields_ = [("left", ctypes.c_void_p), ("right", ctypes.c_void_p), ("stride", ctypes.c_size_t), ("d_init_xy", ctypes.c_void_p),
                        ("ops", ctypes.POINTER(capi.EkfOp)), ("nops", ctypes.c_int), ("nimu", ctypes.c_int)]
        frames = (DevFrame * nframes)()
        keep = []
        for i in range(nframes):
            self.k += 1
            j = frame_index(self.k)
            src = self.ops_dev[self._ekf_inputs(self.k)]
            ops = (capi.EkfOp * self.nops)()
            ctypes.memmove(ops, src, ctypes.sizeof(ops))
            for s_ in range(PREDICTS):
                self.t += 0.005
                ops[2 * s_].t = self.t
            keep.append(ops)
            init = self.d_init[0, j - 1] if j > self.prev_j else self.d_init[1, j]
            fr = frames[i]
            fr.left, fr.right, fr.stride = self.d_frames[j, 0].data_ptr(), (self.d_frames[j, 1].data_ptr() if STEREO else None), W
            fr.d_init_xy, fr.ops, fr.nops, fr.nimu = init.data_ptr(), ops, self.nops, IMU_OPS
            self.prev_j = j
        P = (ctypes.c_void_p * 4)(*[p.h for p in self.pyr])
        ms = ctypes.c_float(0.0)
        drv.hv_dev_run.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.c_void_p] + [ctypes.c_void_p] * 5 + \
                                  [ctypes.c_int, ctypes.POINTER(DevFrame), ctypes.c_int, ctypes.POINTER(ctypes.c_float)]
        capi.check(drv.hv_dev_run(self.ctx.h, self.ctx_b.h, P, self.ekf.h, self.d_points.data_ptr(), self.d_next.data_ptr(), self.d_next2.data_ptr(),
                                  self.d_status.data_ptr(), self.d_ts.data_ptr(), NFEAT, frames, nframes, ctypes.byref(ms)), "hv_dev_run")
        by_handle = {p.h.value: p for p in self.pyr}
        self.pyr = [by_handle[P[i]] for i in range(4)]
        return float(ms.value)

    @staticmethod
    def h2d_bytes():
        return NCAM * W * H + NCAM * NFEAT * 16 + sum(8 * (n * l + 2 * n) for n, l in (ekf_rows(c) for c in range(CHECKS)))

    @staticmethod
    def d2h_bytes():
        return NCAM * NFEAT * 13 + CHECKS * 24 + 8 * (20 + 7 * TRAIL)


def adapter_e2e(inputs, h_frames, which, nframes, warmup):
    """`e2e_adapter`: the step driven through the REFERENCE'S OWN virtual interfaces (tracker::ImagePyramid::Factory / OpticalFlow /
    odometry::EKF) in the order Session::process issues the calls, one synchronous outlier check per track with chiOutlierR, the update
    with visualR, H as a caller-owned Eigen matrix per call (hybvio_b200/host/adapter_e2e_driver.cpp). which = "cuda": the adapters of
    hybvio_b200/host over libhybvio_b200.so; "reference": the reference's own ekf.cpp / OpenCV back ends (same driver source).
    Host buffers in, pose out, wall clock around the loop (the interface is synchronous). Returns None where the library was not
    built (it needs the reference headers at build time)."""
    import ctypes
    path = os.path.join(ROOT, "hybvio_b200", "libhv_adapter_e2e.so") if which == "cuda" else os.path.join(ROOT, "oracle", "_ref", "libref_adapter_e2e.so")
    if not os.path.exists(path):
        return None
    lib = ctypes.CDLL(path)

    class Frame(ctypes.Structure):
        _fields_ = [("left", ctypes.c_void_p), ("right", ctypes.c_void_p), ("init_xy", ctypes.c_void_p), ("imu", ctypes.c_void_p), ("nimu", ctypes.c_int),
                    ("tracks", ctypes.c_void_p), ("track_n", ctypes.c_void_p), ("track_l", ctypes.c_void_p), ("ntracks", ctypes.c_int)]
    total = warmup + nframes
    frames = (Frame * total)()
    tn = np.array([n for _, n, _ in inputs.ekf_off], np.int32)
    tl = np.array([l for _, _, l in inputs.ekf_off], np.int32)
    keep, t, prev_j = [], 0.0, 0
    for i in range(total):
        j = frame_index(i + 1)
        init = np.ascontiguousarray(inputs.init_guess(prev_j, j))
        fr = (i + 1) % POOL_EKF
        imu = np.zeros((PREDICTS, 7))
        for s_ in range(PREDICTS):
            t += 0.005
            imu[s_, 0] = t; imu[s_, 1:] = inputs.imu[fr * PREDICTS + s_]
        keep += [init, imu]
        f = frames[i]
        f.left = h_frames[j, 0].ctypes.data if isinstance(h_frames, np.ndarray) else h_frames[j, 0].data_ptr()
        f.right = None if not STEREO else (h_frames[j, 1].ctypes.data if isinstance(h_frames, np.ndarray) else h_frames[j, 1].data_ptr())
        f.init_xy, f.imu, f.nimu = init.ctypes.data, imu.ctypes.data, PREDICTS
        f.tracks, f.track_n, f.track_l, f.ntracks = inputs.ekf_pool[fr].ctypes.data, tn.ctypes.data, tl.ctypes.data, CHECKS
        prev_j = j
    pose = (ctypes.c_double * 7)()
    ms = ctypes.c_double(0.0)
    counts = (ctypes.c_longlong * 3)()
    lib.hv_adapter_e2e_run.argtypes = [ctypes.c_int] * 5 + [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(Frame)] + [ctypes.c_int] * 3 + \
                                      [ctypes.c_double, ctypes.c_double, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_longlong)]
    pts = np.ascontiguousarray(inputs.points)
    rc = lib.hv_adapter_e2e_run(W, H, NFEAT, MAXLEVEL, TRAIL, pts.ctypes.data, NFEAT, frames, total, warmup, UPDATES, CHI_OUTLIER_R, UPDATE_R, pose,
                                ctypes.byref(ms), counts)
    if rc != 0:
        return {"error": f"hv_adapter_e2e_run returned {rc}"}
    return {"value": round(nframes / (ms.value * 1e-3), 2), "unit": "frames/s", "ms_per_step": round(ms.value / nframes, 5), "steps": nframes,
            "h2d_bytes_per_step": Session.h2d_bytes() if which == "cuda" else 0, "d2h_bytes_per_step": Session.d2h_bytes() if which == "cuda" else 0,
            "calls_per_step": {"outlier_checks": counts[0] / nframes, "inliers": counts[1] / nframes, "updates": counts[2] / nframes,
                               "predict+normalize": PREDICTS, "pyramids": NCAM, "lk": NCAM},
            "pose_finite": bool(np.isfinite(np.array(pose[:])).all()),
            "note": "every call through the reference's virtual interfaces in Session::process order (backend.cpp:729-805, 1158-1185): one synchronous "
                    "visualTrackOutlierCheck per track (its own noise level), updateVisualTrack (a 30x smaller r, the reference's trackChiTestOutlierR : visualR ratio) for the first "
                    f"{UPDATES} inliers, H / f / y as caller-owned Eigen objects per call, host frames in, pose out; wall clock of the calling thread"}


def pin_to_numa_node(node):
    """Pins this process to the host cores of NUMA node `node` (best effort); returns the node or None."""
    try:
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        cpus = [c for c in cpus if c in os.sched_getaffinity(0)]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


def pin_to_gpu_numa_node(torch, local):
    """Pins this process to the host cores of the NUMA node its GPU hangs off (the end-to-end numbers are host-latency bound: a rank on
    the far socket pays for every one of its ~30 synchronous round trips per frame). Best effort; returns the node or None."""
    try:
        bus = torch.cuda.get_device_properties(local).pci_bus_id
        dom = torch.cuda.get_device_properties(local).pci_domain_id
        dev = torch.cuda.get_device_properties(local).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in allowed]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


def gpu_uuid(torch, index):
    """UUID of CUDA device `index` (CUDA_VISIBLE_DEVICES may renumber devices; NVML always sees all of them)."""
    try:
        return str(torch.cuda.get_device_properties(index).uuid)
    except Exception:
        return None


class ClockSampler:
    """SM clock / throttle reasons DURING the timed region (B200_PROFILING.md recipe). The timed region of the default run
    is ~100 ms, shorter than the start-up of an `nvidia-smi -lms` child (which is why earlier lines carried 0 samples), so the
    sampler polls NVML in-process every 10 ms from a thread (the native timed loop releases the GIL); `nvidia-smi` is the
    fallback when NVML cannot be loaded."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index, uuid=None):
        self.rows, self.proc, self.nv, self.th = [], None, None, None
        self.mask, self.sm, self.mx, self.source = 0, [], None, None
        self._stop = threading.Event()
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = None
            if uuid:
                try:
                    h = nv.nvmlDeviceGetHandleByUUID(uuid if str(uuid).startswith("GPU-") else f"GPU-{uuid}")
                except Exception:
                    h = None
            if h is None:
                h = nv.nvmlDeviceGetHandleByIndex(index)
            nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)       # fail here rather than in the thread
            self.mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.nv, self.h, self.source = nv, h, "nvml"
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nv = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi"
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv = self.nv
        reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while True:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.mask |= int(reasons(self.h))
            except Exception:
                pass
            if self._stop.wait(0.010):
                return

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.nv is not None:
            self._stop.set()
            self.th.join(timeout=1.0)
            nv = self.nv
            bits = [nv.nvmlClocksThrottleReasonHwSlowdown, nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                    nv.nvmlClocksThrottleReasonSwThermalSlowdown, nv.nvmlClocksThrottleReasonSwPowerCap]
            reasons = sorted(n for n, b in zip(self.NAMES, bits) if self.mask & int(b))
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.mx, "reasons": reasons,
                    "samples": len(self.sm), "source": "nvml, 10 ms poll"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml and nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        reasons = sorted({self.NAMES[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "source": "nvidia-smi -lms 100"}


def time_kernels(sess, reps=40):
    """Average device time of every launch of one step, CUDA events on the launching stream, inputs cycled through the
    pools. Returns {launch name: {us_per_launch, algo_bytes, gbs, per_step}} in step order."""
    torch = sess.torch
    out = {}

    def timed(name, fn, algo_bytes, per_step=1, stream=None):
        stream = stream or sess.stream
        for i in range(3):
            fn(i)
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            s.record(stream)
            for i in range(reps):
                fn(i + 3)
            e.record(stream)
        e.synchronize()
        us = s.elapsed_time(e) * 1e3 / reps
        out[name] = {"us_per_launch": round(us, 3), "algo_bytes": algo_bytes, "gbs": round(algo_bytes / us * 1e-3, 2), "per_step": per_step}

    inp, ctx, ekf, capi = sess.inp, sess.ctx, sess.ekf, sess.capi
    cur = sess.pyr[2:4]
    N = ekf.N
    timed(f"hv_pyr_fused2_kernel ({NCAM} images)", lambda i: ctx.build_pyramids(cur[:NCAM], [sess.d_frames[(7 * i) % POOL_FRAMES, c] for c in range(NCAM)], device=True),
          NCAM * PYR_BYTES)
    ctx.build_pyramids(cur[:NCAM], [sess.d_frames[1, c] for c in range(NCAM)], device=True)
    ctx.build_pyramids(sess.pyr[0:NCAM], [sess.d_frames[0, c] for c in range(NCAM)], device=True)

    def lk_t(i):
        sess.d_next.copy_(sess.d_init[0, 0])
        ctx.lk_track_device(sess.pyr[0], cur[0], sess.d_points, sess.d_next, sess.d_status, sess.d_ts, NFEAT, True)
    timed("hv_lk_kernel temporal (+ init copy)", lk_t, LK_BYTES)
    if STEREO:
        timed("hv_lk_kernel stereo", lambda i: ctx.lk_track_device(cur[0], cur[1], sess.d_next, sess.d_next2, sess.d_status, sess.d_ts, NFEAT, False), LK_BYTES)

    # ---- rows beyond the step (SURVEY.md 8(f) N2 / N4): reported with per_step = 0, i.e. outside `value` and the roofline shares
    cx_, cy_ = cur[0].gftt_cells(32)
    d_kp = torch.zeros((max(1, cx_ * cy_), 3), dtype=torch.float32, device=sess.dev)
    timed("hv_gftt_kernel (N2 corner detection on level 0; runs when tracks are missing, tracker.cpp:686; not in the step)",
          lambda i: cur[0].gftt_detect_device(d_kp.data_ptr()), W * H + 12 * cx_ * cy_, per_step=0)
    try:
        ing = capi.Ingest(ctx, W, H)
        tab = np.zeros(W * H, np.dtype([("x0", np.int16), ("y0", np.int16), ("xfrac", np.float32), ("yfrac", np.float32)]))
        yy, xx = np.mgrid[0:H, 0:W]
        tab["x0"] = np.clip(xx.ravel(), 0, W - 2); tab["y0"] = np.clip(yy.ravel(), 0, H - 2); tab["xfrac"] = 0.25; tab["yfrac"] = 0.5
        ing.set_remap(tab)
        rgba = torch.from_numpy(np.repeat(sess.h_frames[0, 0].numpy()[:, :, None], 4, axis=2).copy()).pin_memory()
        lib_ = capi.load()

        def ingest(i):
            capi.check(lib_.hv_ingest_frame(ing.h_, rgba.data_ptr(), 4 * W, 4, None, cur[0].h, None), "hv_ingest_frame")
        timed("hv_ingest_frame (N4: RGBA frame H2D + hv_gray_kernel + hv_remap_kernel + pyramid in place; not in the step)", ingest,
              4 * W * H + 5 * W * H + 14 * W * H + PYR_BYTES, per_step=0)
        ctx.sync(); ing.close()
        ctx.build_pyramids(cur[:NCAM], [sess.d_frames[1, c] for c in range(NCAM)], device=True)
    except Exception as ex:      # noqa: BLE001 -- report-only row
        out["hv_ingest_frame (N4)"] = {"error": repr(ex)[:200], "per_step": 0, "us_per_launch": 0.0, "algo_bytes": 0, "gbs": 0.0}

    def pred(i):
        ops = sess.ops_dev[i % POOL_EKF]
        for s_ in range(PREDICTS):
            sess.t += 0.005
            ops[2 * s_].t = sess.t
        ekf.run_device(ops, IMU_OPS)
        ekf.flush()
    B = sess.stream_b
    timed(f"ekf_predict_kernel ({PREDICTS} samples + normalisations, one launch)", pred, PREDICTS * 2 * 8 * (40 * N - 400), stream=B)
    for c in range(UPDATES):
        n, l = ekf_rows(c)

        def upd(i, c=c):
            ops = sess.ops_dev[i % POOL_EKF]
            ekf.run_device(ctypes_slice(ops, IMU_OPS + c, 1), 1)
        timed(f"ekf_update_cluster2_kernel check+update #{c} (n={n},l={l})", upd, 2 * 8 * N * N + 8 * n * l, stream=B)
        ekf.symmetrize(); ekf.augment(-1)

    def chk(i):
        ops = sess.ops_dev[i % POOL_EKF]
        ekf.run_device(ctypes_slice(ops, IMU_OPS + UPDATES, CHECKS - UPDATES), CHECKS - UPDATES)
    timed(f"ekf_check_batch_cluster2_kernel ({CHECKS - UPDATES} tracks, one cluster each)", chk,
          sum(8 * N * N + 8 * n * l for n, l in (ekf_rows(c) for c in range(UPDATES, CHECKS))), stream=B)
    def sym_aug(i):
        ekf.symmetrize(); ekf.augment(-1)
    timed("ekf_update_cluster2_kernel symmetrise + augment (one launch)", sym_aug, 2 * 8 * N * N, stream=B)
    return out


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(sess, out_dir):
    """--dump-outputs: what the last frame of the timed device-resident loop handed its caller, as float32 / float64 arrays in
    out_dir/<name>.npy -- optical-flow end points and statuses, the frame's pyramids, the outlier decisions of its visual updates
    and the filter state after the augmentation. The inputs are seeded, so two builds run with the same arguments can be compared
    file by file."""
    sess.torch.cuda.synchronize()
    out = {"lk_temporal_next_xy": sess.d_next.cpu().numpy()}
    if STEREO:
        out["lk_stereo_next_xy"] = sess.d_next2.cpu().numpy()
    # both LK calls of a frame write the same status buffers: these are the last call's (the stereo one where there is one)
    out["lk_status"] = sess.d_status.cpu().numpy().astype(np.float32)
    out["lk_track_status"] = sess.d_ts.cpu().numpy().astype(np.float32)
    for c, side in enumerate(("left", "right")[:NCAM]):
        pyr = sess.pyr[c]                      # the loop has rotated the frame's pyramids into the "previous frame" slots
        for lv in range(pyr.levels):
            gray, grad = pyr.download(lv)
            out[f"pyramid_{side}_gray_l{lv}"] = gray.astype(np.float32)
            out[f"pyramid_{side}_grad_l{lv}"] = grad.astype(np.float32)
    status, chi2 = sess.ekf.run_device_results(sess.nops - IMU_OPS)
    out["ekf_outlier_status"] = status[:CHECKS].astype(np.float64)
    out["ekf_chi2"] = chi2[:CHECKS]
    m, P = sess.ekf.download()
    out["ekf_mean"] = m
    out["ekf_covariance"] = np.ascontiguousarray(P)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes (limit {DUMP_MAX_BYTES})")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def ctypes_slice(arr, start, count):
    import ctypes
    return ctypes.cast(ctypes.byref(arr, start * ctypes.sizeof(arr._type_)), ctypes.POINTER(arr._type_))


def time_batched(sess, reps=20):
    """What the same kernels reach when one launch carries many independent sessions (pyramid: 32 images, LK: 8 jobs x
    150 features): shows how far the single-session numbers are from the kernels' own limits."""
    torch = sess.torch
    out = {}
    ctx = sess.ctx
    pyrs = [ctx.pyramid(W, H, WIN, MAXLEVEL) for _ in range(32)]
    imgs = [sess.d_frames[(3 * i) % POOL_FRAMES, i % 2] for i in range(32)]

    def run(name, fn, algo):
        for _ in range(3):
            fn()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(sess.stream):
            s.record(sess.stream)
            for _ in range(reps):
                fn()
            e.record(sess.stream)
        e.synchronize()
        us = s.elapsed_time(e) * 1e3 / reps
        out[name] = {"us_per_launch": round(us, 2), "algo_bytes": algo, "gbs": round(algo / us * 1e-3, 1)}
    run("hv_pyr_fused2_kernel (32 images, one launch)", lambda: ctx.build_pyramids(pyrs, imgs, device=True), 32 * PYR_BYTES)
    capi = sess.capi
    jobs = (capi.LkJob * 8)()
    bufs = []
    for j in range(8):
        nxt = torch.zeros((NFEAT, 2), dtype=torch.float32, device=sess.dev); st = torch.zeros(NFEAT, dtype=torch.uint8, device=sess.dev)
        bufs += [nxt, st]
        jobs[j].prev, jobs[j].next = pyrs[2 * j].h, pyrs[2 * j + 1].h
        jobs[j].d_prev_xy, jobs[j].d_next_xy, jobs[j].d_status, jobs[j].d_track_status = sess.d_points.data_ptr(), nxt.data_ptr(), st.data_ptr(), None
        jobs[j].n, jobs[j].use_initial = NFEAT, 0
    lib = capi.load()
    run("hv_lk_kernel (8 sessions x 150 features, one launch)", lambda: capi.check(lib.hv_lk_track_batch_device(ctx.h, jobs, 8, 20, 0.03, 1e-3), "lk batch"), 8 * LK_BYTES)
    ctx.sync()
    for p in pyrs:
        p.release()
    return out


def aggregate_ms(ms_local, device, world):
    """Device time of the step loop = MAX over ranks (each rank runs its own independent session)."""
    import torch
    import torch.distributed as dist
    ms = torch.tensor([ms_local], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


def frames_per_second(world, steps, ms):
    """Whole-job throughput: every rank processed `steps` frames of its own session in `ms` (weak scaling)."""
    return world * steps / (ms * 1e-3)


def run_selftest_dist(args):
    """CPU-only check of the multi-process plumbing (gloo): rank r pretends its loop took (10 + r) ms."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0"))
    if world > 1:
        dist.init_process_group("gloo")
        dist.barrier()
    ms = aggregate_ms(10.0 + rank, torch.device("cpu"), world)
    if world > 1:
        dist.barrier(); dist.destroy_process_group()
    if rank == 0:
        emit(json.dumps({"selftest": True, "n_gpus": world, "ms": ms, "value": frames_per_second(world, args.steps, ms), "scaling": "weak"}))


def run_ours(args):
    if args.sessions > 1:
        # several sessions share the GPU: a dependent kernel that was launched early (programmatic dependent launch) would hold
        # an SM and ~200 KB of shared memory while it waits for its predecessor -- SMs the other sessions could use
        os.environ.setdefault("HV_EKF_NO_PDL", "1")
        # ... and every session brings its own streams: with the default of 8 hardware work queues they alias, so that a kernel of one
        # session queues behind an unrelated one of another (measured, 8 sessions: 11,080 frames/s with 8 queues, 22,820 with 32)
        os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device. hybvio_b200 has no CPU fallback; use --impl reference for the CPU arm.")
    torch.cuda.set_device(local)
    os.environ["HV_DEVICE"] = str(local)              # the C++ adapters (e2e_adapter) work on this rank's GPU, not on GPU 0
    numa_node = pin_to_gpu_numa_node(torch, local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    inputs = Inputs(torch.device("cuda", local), seed=rank)
    nsess = max(1, args.sessions)
    sessions = [Session(local, inputs) for _ in range(nsess)]      # independent sessions on this GPU (own streams, pyramids, EKF)
    sess = sessions[0]

    def run_parallel(fn_name, nframes):
        """Runs sessions[i].<fn_name>(nframes) concurrently, one host thread per session (the native drivers release the GIL);
        returns the largest per-session device time: all sessions start together, the job is done when the slowest one is."""
        if nsess == 1:
            r = getattr(sess, fn_name)(nframes)
            return r[0] if isinstance(r, tuple) else r
        out = [0.0] * nsess
        gate = threading.Barrier(nsess)

        def work(i):
            torch.cuda.set_device(local)
            gate.wait()
            r = getattr(sessions[i], fn_name)(nframes)
            out[i] = r[0] if isinstance(r, tuple) else r
        th = [threading.Thread(target=work, args=(i,)) for i in range(nsess)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        return max(out)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_loop(step, steps, warmup):
        for _ in range(warmup):
            step()
        barrier()
        sampler = ClockSampler(local, gpu_uuid(torch, local)) if rank == 0 else None
        launches0 = sess.ctx.launches + sess.ctx_b.launches
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(sess.stream)
        for _ in range(steps):
            step()
        sess.ctx_b.sync()                          # EKF stream and the library's side stream (outlier checks of the last frames)
        sess.stream.wait_stream(sess.stream_b)
        e.record(sess.stream)
        e.synchronize()
        barrier()
        ms = aggregate_ms(s.elapsed_time(e), sess.dev, world)
        clocks = sampler.stop() if sampler else None
        return ms, sess.ctx.launches + sess.ctx_b.launches - launches0, clocks

    def launch_count():
        return sum(x.ctx.launches + x.ctx_b.launches for x in sessions)

    with torch.cuda.stream(sess.stream):
        # value: device-resident loop issued by the native caller (hv_dev_run); the Python-driven variant of the same calls
        # (step_device) is reported next to it as python_harness
        ms_dev_py, _, _ = timed_loop(sess.step_device, min(args.steps, 100), args.warmup)
        run_parallel("run_dev_native", args.warmup)
        barrier()
        sampler = ClockSampler(local, gpu_uuid(torch, local)) if rank == 0 else None
        launches0 = launch_count()
        ms_local = run_parallel("run_dev_native", args.steps)
        launches = launch_count() - launches0
        clocks = sampler.stop() if sampler else None
        barrier()
        ms_dev = aggregate_ms(ms_local, sess.dev, world)
        if args.dump_outputs and rank == 0:
            dump_outputs(sess, args.dump_outputs)
        if args.step_only:
            if rank == 0:
                emit(json.dumps({"metric": METRIC(), "value": round(frames_per_second(world * nsess, args.steps, ms_dev), 2), "steps": args.steps,
                                  "warmup": args.warmup, "gpu_launches": launches, "note": "--step-only: device-resident loop only, no e2e / kernel rows"}))
            return
        e2e_steps = max(3, min(args.steps, args.e2e_steps))
        # e2e: native caller of the host-buffer C ABI (hybvio_b200/host/e2e_driver.cu); the Python-driven variant of the
        # same calls (step_e2e) is reported next to it as e2e.python_harness
        ms_e2e_py, _, _ = timed_loop(sess.step_e2e, e2e_steps, max(3, min(args.warmup, 10)))
        run_parallel("run_e2e_native", max(3, min(args.warmup, 10)))
        barrier()
        ms_native = run_parallel("run_e2e_native", e2e_steps)
        barrier()
        ms_e2e = aggregate_ms(ms_native, sess.dev, world)
        m, P = sess.ekf.download()
        healthy = bool(np.isfinite(m).all() and np.isfinite(P).all() and (np.diag(P) >= 0).all())
        barrier()
        # e2e_adapter: every rank runs it (own GPU, own host thread), the slowest rank counts
        ad = adapter_e2e(inputs, sess.h_frames, "cuda", max(20, min(e2e_steps, 200)), 10) if nsess == 1 else None
        ad_ms = aggregate_ms(ad["ms_per_step"] if ad and "ms_per_step" in ad else 0.0, sess.dev, world)
        barrier()
        kern = time_kernels(sess) if rank == 0 else None
        kbatch = time_batched(sess) if rank == 0 else None

    result = None
    if rank == 0:
        value = frames_per_second(world * nsess, args.steps, ms_dev)
        e2e = frames_per_second(world * nsess, e2e_steps, ms_e2e)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)") if "hbm_gbs" in peaks else (6650.0, "fallback (B200_PROFILING.md)")
        shares = {k: v["us_per_launch"] * v["per_step"] for k, v in kern.items()}
        tot = sum(shares.values())
        fam = {}
        for k, v in shares.items():
            fam[k.split(" ")[0]] = fam.get(k.split(" ")[0], 0.0) + v
        domfam = max(fam, key=lambda k: fam[k])
        dom = max((k for k in shares if k.startswith(domfam)), key=lambda k: shares[k])
        traffic = None
        try:   # dram__bytes_read.sum + dram__bytes_write.sum of the same launch from the committed ncu --set full capture
            name = "r02_ncu_full_summary.json" if os.path.exists(os.path.join(ROOT, "profiles", "r02_ncu_full_summary.json")) else "r01_ncu_full_summary.json"
            prof = json.load(open(os.path.join(ROOT, "profiles", name)))
            key = "check+update n=84" if "n=84" in dom else "augment" if "augment" in dom else None
            traffic = next((int(e["dram_bytes"]) for e in prof["kernels"] if key and key in e["launch"]), None)
        except Exception:
            pass
        roof = {"bound": "hbm", "kernel": dom, "achieved": kern[dom]["gbs"], "peak": peak, "unit": "GB/s", "frac": round(kern[dom]["gbs"] / peak, 5),
                "traffic": traffic, "peak_source": peak_src, "share_of_step": round(shares[dom] / tot, 3),
                "kernel_family_share_of_step": {k: round(v / tot, 3) for k, v in fam.items()},
                "note": "achieved = algorithmic bytes (SURVEY.md 8(d)) / CUDA-event launch time of the largest launch of the kernel with the largest "
                        "share of the step; one VIO session is a chain of small dependent launches (latency-bound), see DESIGN.md 4 and kernels_batched"}
        if "n=84" in dom:
            # what actually bounds this kernel: fp64 tensor-core (DMMA) work on the 8 SMs of its cluster + the serial pivot chain
            n_, l_, N_ = 84, 160, sess.ekf.N
            fma = n_ * l_ * N_ + n_ * n_ * l_ / 2 + n_ ** 3 / 3 + n_ * n_ * (N_ + 1) / 2 + N_ * N_ * n_
            gf = 2 * fma / kern[dom]["us_per_launch"] * 1e-3
            peak8 = 64 * 2 * 1.965 * 8      # 64 FMA/clk/SM (tools/probe2.cu) x 2 flop x 1.965 GHz x 8 SMs, GFLOP/s
            roof["fp64_tensor"] = {"fma_per_launch": int(fma), "achieved_gflops": round(gf, 1), "peak_gflops_of_the_8_sms_used": round(peak8, 1),
                                   "frac": round(gf / peak8, 4), "note": "DMMA m8n8k4 measured at 64 FMA/clk/SM on B200; the kernel runs on one 8-CTA cluster"}
        for k in kern:
            kern[k]["frac_of_hbm_peak"] = round(kern[k]["gbs"] / peak, 5)
            kern[k]["share_of_step"] = round(shares[k] / tot, 3)
        for k in kbatch:
            kbatch[k]["frac_of_hbm_peak"] = round(kbatch[k]["gbs"] / peak, 5)
        result = {
            "metric": METRIC(), "value": round(value, 2), "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_dev / args.steps, 5), "higher_is_better": True,
            "python_harness": {"value": round(frames_per_second(world, min(args.steps, 100), ms_dev_py), 2),
                               "note": "the same device-resident frames issued call by call from Python (one session)"},
            "scaling": "weak", "vs_baseline": None, "dtype": "u8/s16 fixed-point + f32 (pyramid, LK), f64 (EKF)", "data": "synthetic",
            "config": {"workload": CONFIG_NAME + f"; per frame {NCAM} pyramid(s) + {NCAM} LK call(s) + 10 x (predict + normalizeQuaternions(true)) + "
                                   f"20 checks (5 with update, n = {'/'.join(map(str, N_ROWS))} rows) + symmetrise + augment; independent sessions, " + str(nsess) + " per GPU",
                       "baseline_config": CONFIG_ID, "host_numa_node_pinned": numa_node,
                       "sessions_per_gpu": nsess,
                       "streams": "per session: pyramid builds on the tracker stream; mean propagation -> LK(k) -> visual updates(k) -> augmentation in stream order on the filter stream (the flow predictor reads the propagated pose); covariance propagation and the outlier checks that precede the augmentation on streams of the library",
                       "l2": f"inputs cycled through pools larger than L2 (frames {POOL_FRAMES * 2 * W * H / 1e6:.0f} MB + EKF inputs "
                             f"{POOL_EKF * inputs.ekf_stride * 8 / 1e6:.0f} MB > 126 MB); no explicit flush",
                       "ekf_healthy_after_run": healthy},
            "e2e": {"value": round(e2e, 2), "unit": "frames/s", "h2d_bytes_per_step": Session.h2d_bytes(), "d2h_bytes_per_step": Session.d2h_bytes(),
                    "steps": e2e_steps, "ms_per_step": round(ms_e2e / e2e_steps, 5),
                    "host_phase_us_per_step": sess.e2e_host_phase_us,
                    "python_harness": {"value": round(frames_per_second(world, e2e_steps, ms_e2e_py), 2), "ms_per_step": round(ms_e2e_py / e2e_steps, 5)},
                    "note": "host-buffer C ABI driven by a native caller (host/e2e_driver.cu): pinned H2D of both frames, synchronous LK results, every check+update and the batched checks return to the host, pose read-back"},
            "e2e_adapter": (dict(ad, value=round(world * 1e3 / ad_ms, 2), ms_per_step=round(ad_ms, 5)) if ad and "ms_per_step" in ad else
                            (ad or {"unavailable": "hybvio_b200/libhv_adapter_e2e.so not built (needs the reference headers at build time) or --sessions > 1"})),
            "gpu_launches": int(launches), "gpu_launches_per_step": round(launches / (args.steps * nsess), 2),
            "clocks": clocks, "roofline": roof, "kernels": kern, "kernels_batched": kbatch,
        }
        if world == 1 and not args.no_cpu_baseline:
            result["cpu_baseline"] = cpu_baseline(inputs, budget_s=args.cpu_budget)
        if world == 1 and nsess == 1 and CONFIG_ID == 2 and not os.environ.get("HV_BENCH_CHILD"):
            for key, extra in (("next_row_track_model", next_row_track_model),):
                elapsed = time.monotonic() - T_PROCESS_START
                if os.environ.get("HV_BENCH_NO_EXTRAS"):
                    result[key] = {"skipped": "HV_BENCH_NO_EXTRAS"}
                elif elapsed > EXTRAS_START_BY:
                    result[key] = {"skipped": f"time budget: {elapsed:.0f} s into the run (limit {EXTRAS_START_BY:.0f} s)"}
                else:
                    result[key] = extra()
            # e2e_chain: the frame with the WHOLE visual-update loop of backend.cpp:1012-1252 on both sides -- triangulation + prepareVisualUpdate +
            # outlier check + update per track (here: hv_ekf_visual_tracks, 20 candidate tracks, 5 updates, one host synchronisation; reference:
            # its own triangulation.cpp + ekf.cpp on one host thread) -- composed from parts measured in this run: tracker phases of the e2e loop
            # (host buffers, synchronous LK), the IMU burst and the augmentation launch, and the loop as timed by tests/tools/track_model_bench.py
            tm = result.get("next_row_track_model") or {}
            loop = (tm.get("visual_update_loop") or {})
            cb = result.get("cpu_baseline") or {}
            if loop.get("chain_one_sync_us") and kern:
                hp = sess.e2e_host_phase_us
                pred = next((v["us_per_launch"] for k_, v in kern.items() if k_.startswith("ekf_predict")), 0.0)
                aug = next((v["us_per_launch"] for k_, v in kern.items() if "augment" in k_), 0.0)
                ours_us = hp["pyramids_submit"] + hp["lk_temporal"] + hp["lk_stereo"] + pred + loop["chain_one_sync_us"] + aug
                entry = {"value": round(1e6 / ours_us, 2), "unit": "frames/s", "us_per_step": round(ours_us, 1),
                         "parts_us": {"tracker_host_phases": round(hp["pyramids_submit"] + hp["lk_temporal"] + hp["lk_stereo"], 1), "imu_burst_launch": pred,
                                      "visual_update_loop (hv_ekf_visual_tracks, 20 tracks, 5 updates, one sync)": loop["chain_one_sync_us"], "symmetrise+augment": aug},
                         "h2d_bytes_per_step": NCAM * W * H + NCAM * NFEAT * 16 + 20 * 1400, "d2h_bytes_per_step": NCAM * NFEAT * 13 + 20 * 64 + 16,
                         "same_decisions_as_cpu_reference": loop.get("same_decisions_as_cpu_reference"),
                         "note": "COMPOSED from parts measured in this run, not one timed loop; H never leaves the device (the track observations go up: ~1.4 KB per track)"}
                st = (cb.get("stage_ms_per_frame") or {})
                cpu_loop = (loop.get("cpu_reference_loop") or {}).get("us")
                if st and cpu_loop:
                    ref_us = 1e3 * (st.get("pyramid", 0) + st.get("lk", 0) + st.get("ekf_predict", 0) + st.get("ekf_augment", 0)) + cpu_loop
                    entry["reference"] = {"value": round(1e6 / ref_us, 2), "unit": "frames/s", "us_per_step": round(ref_us, 1),
                                          "note": "reference pyramid + LK + predict + augment stage times of cpu_baseline + its own triangulation.cpp / ekf.cpp loop on one host thread"}
                result["e2e_chain"] = entry
    for x in sessions:
        x.ctx.sync(); x.ctx_b.sync()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        emit(json.dumps(result))


def next_row_track_model():
    """SURVEY.md 8(f) N1 (triangulation + prepareVisualUpdate on the device): measured and checked against the oracle by
    tests/tools/track_model_bench.py in a SEPARATE process after the headline measurement, so that nothing it does can disturb
    the line above; not part of value / e2e."""
    import subprocess
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "tools", "track_model_bench.py")], capture_output=True, text=True, timeout=EXTRAS_TIMEOUT)
        lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
        if lines:                                         # the tool prints its line before it tears the context down
            d = json.loads(lines[-1])
            if r.returncode != 0:
                d["exit_code"] = r.returncode
            return d
        return {"error": (r.stderr or r.stdout)[-400:]}
    except Exception as ex:       # noqa: BLE001 -- a report-only extra must never take the bench line down
        return {"error": repr(ex)[:400]}


# ------------------------------------------------------------------------------------------------ reference arm
class RefSession:
    """The reference's own CPU path for the same step: vendored OpenCV 4.3 pyramid + LK (oracle/_ref/libref_lk.so,
    OpenCV pthreads on all cores) and src/odometry/ekf.cpp (oracle/_ref/libref_ekf.so, single thread like the
    reference build's -DEIGEN_DONT_PARALLELIZE). Falls back to the C port (oracle/) where _ref was not built."""

    def __init__(self, inputs):
        import ctypes
        from oracle import ekf_oracle, lk_oracle
        self.inp = inputs
        self.frames = inputs.frames.cpu().numpy()
        if lk_oracle.have_ref() and ekf_oracle.have_ref():
            self.kind, self.lk = "reference", lk_oracle.RefLK()
            make_ekf = ekf_oracle.RefEKF
            self.cores = self.lk.threads
        else:
            if not os.path.exists(lk_oracle.ORACLE_SO):
                subprocess.check_call(["make", "-C", ROOT, "oracle"])
            self.kind, self.lk = "port", lk_oracle.OracleLK()
            make_ekf = ekf_oracle.OracleEKF
            self.cores = 1
        e = make_ekf()
        p = e.default_params(); p.camera_trail_length = TRAIL
        e.close()
        self.ekf = make_ekf(p)
        self.pyr = [self.lk.pyramid(self.frames[0, i % 2], WIN, MAXLEVEL) for i in range(4)]
        self.t, self.k, self.prev_j = 0.0, 0, 0
        self.ekf.initialize_orientation(inputs.imu[0, 3:])

    STAGES = ("pyramid", "lk", "ekf_predict", "ekf_check", "ekf_update", "ekf_augment")

    def step(self, stage_s=None):
        """One stereo frame. stage_s: optional dict that accumulates wall-clock seconds per stage (SURVEY.md 8(d) per-stage rows)."""
        clock = time.perf_counter
        t_ = clock()

        def lap(name):
            nonlocal t_
            if stage_s is not None:
                now = clock()
                stage_s[name] = stage_s.get(name, 0.0) + now - t_
                t_ = now

        self.k += 1
        j = frame_index(self.k)
        inp = self.inp
        cur = self.pyr[2:4]
        if self.kind == "reference":
            for c_ in range(NCAM):
                self.lk.rebuild(cur[c_], self.frames[j, c_])
        else:
            for q in cur[:NCAM]:
                q.free()
            cur = [self.lk.pyramid(self.frames[j, c_], WIN, MAXLEVEL) for c_ in range(NCAM)] + cur[NCAM:]
            self.pyr[2:4] = cur
        lap("pyramid")
        nxt, st, ts = self.lk.lk(self.pyr[0], cur[0], inp.points, inp.init_guess(self.prev_j, j), max_level=MAXLEVEL)
        if STEREO:
            nxt2, st2, ts2 = self.lk.lk(cur[0], cur[1], nxt, None, max_level=MAXLEVEL)
        lap("lk")
        fr = self.k % POOL_EKF
        for s in range(PREDICTS):
            self.t += 0.005
            u = inp.imu[fr * PREDICTS + s]
            self.ekf.predict(self.t, u[:3], u[3:])
            self.ekf.normalize_quaternions(True)
        lap("ekf_predict")
        row = inp.ekf_pool[fr]
        for c, (o, n, l) in enumerate(inp.ekf_off):
            Hm = row[o:o + n * l].reshape((n, l), order="F")
            f, y = row[o + n * l:o + n * l + n], row[o + n * l + n:o + n * l + 2 * n]
            st_, _ = self.ekf.visual_check(Hm, f, y, VISUAL_R)
            lap("ekf_check")
            if c < UPDATES and st_ == 0:
                self.ekf.visual_update(Hm, f, y, VISUAL_R)
                lap("ekf_update")
        self.ekf.symmetrize()
        self.ekf.augment(-1)
        lap("ekf_augment")
        self.pyr = self.pyr[2:4] + self.pyr[0:2]
        self.prev_j = j


def cpu_baseline(inputs, budget_s=12.0):
    rs = RefSession(inputs)
    for _ in range(5):
        rs.step()
    t0 = time.perf_counter()
    for _ in range(10):
        rs.step()
    per = (time.perf_counter() - t0) / 10
    n = int(max(20, min(1500, budget_s / per)))
    t0 = time.perf_counter()
    for _ in range(n):
        rs.step()
    dt = time.perf_counter() - t0
    # per-stage rows (SURVEY.md 8(d)): a short instrumented pass after the timed one, so that the timers are not inside `value`
    stage_s, m = {}, max(10, min(100, n // 10))
    for _ in range(m):
        rs.step(stage_s)
    stages = {k: round(stage_s.get(k, 0.0) / m * 1e3, 4) for k in RefSession.STAGES}
    stages["frame_total"] = round(sum(stage_s.values()) / m * 1e3, 4)
    one_thread = None
    if rs.kind == "reference" and hasattr(rs.lk, "set_threads"):       # the cv::setNumThreads(1) row of SURVEY.md 8(d)
        all_threads = rs.cores
        try:
            rs.lk.set_threads(1)
            s1, m1 = {}, max(5, m // 2)
            for _ in range(m1):
                rs.step(s1)
            one_thread = {"pyramid": round(s1.get("pyramid", 0.0) / m1 * 1e3, 4), "lk": round(s1.get("lk", 0.0) / m1 * 1e3, 4),
                          "frame_total": round(sum(s1.values()) / m1 * 1e3, 4)}
        finally:
            rs.lk.set_threads(all_threads)
    ad = adapter_e2e(inputs, rs.frames, "reference", 60, 10) if rs.kind == "reference" else None
    return {"value": round(n / dt, 2), "unit": "frames/s", "cores": rs.cores, "kind": rs.kind, "host_cores": os.cpu_count(),
            "e2e_adapter": ad or {"unavailable": "oracle/_ref/libref_adapter_e2e.so not built"},
            "sample": f"{n} consecutive stereo frames of the same workload ({dt:.1f} s); pyramid+LK on {rs.cores} OpenCV threads, EKF on 1 thread "
                      f"(reference builds Eigen with EIGEN_DONT_PARALLELIZE)",
            "stage_ms_per_frame": stages, "stage_ms_per_frame_one_opencv_thread": one_thread,
            "stage_sample": f"{m} instrumented frames after the timed ones"}


def run_reference(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0"))) if torch.cuda.is_available() else torch.device("cpu")
    # The reference gets the same host placement as our arm: the cores of ONE NUMA node (the GPU's, or node 0). Measured on the 2-socket B200
    # hosts: OpenCV's thread pool spread over both sockets needs 3.5 ms per pyramid pair and 4.9 ms per LK pair, pinned to one socket 0.67 /
    # 0.32 ms -- unpinned the reference arm ran at 80 frames/s, pinned at 139.
    numa_node = pin_to_gpu_numa_node(torch, int(os.environ.get("LOCAL_RANK", "0"))) if torch.cuda.is_available() else pin_to_numa_node(0)
    inputs = Inputs(dev, seed=0)       # torch is only the synthetic-input generator here; the timed path is pure CPU
    rs = RefSession(inputs)
    # >= 50 warm-up frames whatever --warmup says: OpenCV's thread pool, the page cache of the frame pool and the CPU clocks need them
    # (round 1: 76 frames/s after 5 warm-up frames against 89-123 over 1000+ frames)
    ref_warmup = max(50, args.warmup)
    for _ in range(ref_warmup):
        rs.step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        rs.step()
    dt = time.perf_counter() - t0
    v = args.steps / dt
    stage_s, m = {}, max(5, min(50, args.steps))              # per-stage rows from a few instrumented frames AFTER the timed ones
    for _ in range(m):
        rs.step(stage_s)
    stages = {k: round(stage_s.get(k, 0.0) / m * 1e3, 4) for k in RefSession.STAGES}
    ad = adapter_e2e(inputs, rs.frames, "reference", max(20, min(args.steps, 100)), 10)
    emit(json.dumps({
        "impl": "reference", "metric": METRIC(), "value": round(v, 2), "unit": "frames/s", "n_gpus": world,
        "steps": args.steps, "warmup": ref_warmup, "ms_per_step": round(dt / args.steps * 1e3, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8/s16 fixed-point + f32 (pyramid, LK), f64 (EKF)", "data": "synthetic",
        "config": {"workload": CONFIG_NAME + " (same step as the CUDA arm) on the host CPU; ONE session on rank 0 whatever --gpus says",
                   "baseline_config": CONFIG_ID, "host_numa_node_pinned": numa_node},
        "sessions": 1,
        "e2e_adapter": ad or {"unavailable": "oracle/_ref/libref_adapter_e2e.so not built"},
        "cpu_baseline": {"value": round(v, 2), "unit": "frames/s", "cores": rs.cores, "kind": rs.kind, "host_cores": os.cpu_count(),
                         "sample": f"{args.steps} stereo frames", "stage_ms_per_frame": stages},
        "e2e": {"value": round(v, 2), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


_REAL_STDOUT = None


def claim_stdout():
    """Only the final JSON line may reach stdout: libraries (NCCL prints its version banner there) are redirected to
    stderr for the whole run."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    _REAL_STDOUT.write(line + "\n")
    _REAL_STDOUT.flush()


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=200)
    ap.add_argument("--sessions", type=int, default=1, help="independent VIO sessions per GPU (default 1 = BASELINE config 2; config 3 shares a GPU between streams when G < 8)")
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="BASELINE.json config: 2 (default, the headline), 4 (512x512, 200 features, N=62), 1 (mono)")
    ap.add_argument("--step-only", action="store_true", help="only the device-resident timed loop (for `ncu` launch lists of the step: profiles/README.md)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed (end points, statuses, "
                                                           "pyramids, outlier decisions, filter state) as DIR/<name>.npy (CUDA arm)")
    ap.add_argument("--selftest-dist", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA arm (--impl ours)")
    args.warmup = max(3, args.warmup)
    set_config(args.config)
    if args.selftest_dist:
        run_selftest_dist(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
