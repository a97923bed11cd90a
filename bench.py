#!/usr/bin/env python
"""bench.py — frames/sec of the VINS-Mono hot path (feature tracker + sliding-window BA) on B200.

A "step" is one published (10 Hz) frame of one sequence, fully processed: the two 752x480 camera images that
arrive in that interval go through FeatureTracker::readImage (the second one publishes), the ~20 IMU samples
through processIMU, the feature message through Estimator::processImage (triangulate, 8-iteration dogleg solve,
marginalisation, slide).  Inputs are synthetic (harness/synth.py), no dataset is read.

Workloads (BASELINE.json configs):
  N = 1 (default)   configs[1]: one sequence on the GPU (the headline line); the same line carries a "c3" object =
                    configs[2], 64 independent sequences on the same GPU through the batched path
  N > 1 (torchrun)  configs[4]'s share per GPU: 64 sequences per rank (512 on 8 GPUs), no data-path collective
  --config c3       emit the configs[2] line as the main line on one GPU

  python bench.py [--gpus N] [--steps K] [--warmup W]            our CUDA path
  python bench.py ... --dump-outputs DIR                          also write the last timed step's outputs as DIR/*.npy
  python bench.py --impl reference ...                            the CPU path: cv2 (OpenCV) tracker twin + oracle estimator
Under torchrun (N > 1) rank 0 prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from harness import synth, pipeline  # noqa: E402

METRIC = "frames/sec (tracker+BA) at 752x480, 10-KF window, 150 feats; ATE vs ref"
WORKLOAD = ("configs[1]: single 752x480 synthetic sequence per GPU, 10-keyframe window, 150 features, 200 Hz IMU, "
            "fp64 Jacobians")
WORKLOAD_BATCH = ("configs[2]/[4]: {s} independent 752x480 synthetic sequences per GPU ({d} distinct trajectories/scenes, "
                  "replicated), 10-keyframe window, 150 features, 200 Hz IMU, fp64 Jacobians, batched launches")
INIT_PUBS = 12           # published frames consumed before the window is full and seeded (estimator goes NON_LINEAR)
ALGO_BYTES_IMAGE = 1_319_760   # SURVEY.md §8(d): compulsory front-end traffic per input image
ALGO_BYTES_SOLVE = 233_000     # SURVEY.md §8(d): back-end inputs+outputs per solve at C1
SEQS_PER_GPU = 64
# estimator / tracker parameters of the workload (configs[3] swaps them: see main)
TRK_KW = {}
EST_KW = {}
ORC_KW = {}
WORKLOAD_C4 = ("configs[3]: single 752x480 synthetic sequence, 20-keyframe window, 300 features (min_dist 20), ProjectionTdFactor with "
               "estimate_td and rolling-shutter row term (TR 0.033 s), 200 Hz IMU, fp64 Jacobians")


def sequence_inputs(seed, n_pub):
    """Rendered frames + IMU of one sequence, enough for n_pub published frames."""
    n_img = 2 * (n_pub + 1) + 2
    seq = synth.Sequence(seed=seed, duration=n_img / 20.0 + 0.5)
    ts, imgs = pipeline.cached_images(seq, n_img)
    t_imu, acc, gyr = seq.imu()
    return seq, ts, np.ascontiguousarray(imgs), (t_imu, acc, gyr)


class BatchedImu(pipeline.ImuFeeder):
    """Same sample selection / interpolation as estimator_node.cpp:98-136, 225-265, delivered in one call."""

    def feed(self, estimator, stamp, td=None):
        rec = _Recorder()
        super().feed(rec, stamp, estimator.states()[1] if td is None else td)
        if rec.dt:
            estimator.processIMU_batch(np.array(rec.dt), np.array(rec.acc), np.array(rec.gyr))


class _Recorder:
    def __init__(self):
        self.dt, self.acc, self.gyr = [], [], []

    def processIMU(self, dt, a, g):
        self.dt.append(dt)
        self.acc.append(np.array(a, float))
        self.gyr.append(np.array(g, float))


class ClockSampler:
    """SM clock and throttle reasons polled through NVML (every ~2 ms) while a pass runs; the reported figures use the
    samples that fall inside the timed region (SoloGate marks its begin / end)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index, self.rows, self.stop_flag, self.thread = index, [], threading.Event(), None
        self.t_begin = self.t_end = None
        self.max_mhz = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES-agnostic lookup is not needed: one process per GPU with LOCAL_RANK == device index
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception:  # no NVML: report nothing rather than fail the bench
            return

        def poll():
            while not self.stop_flag.is_set():
                try:
                    mhz = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                    why = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    self.rows.append((time.perf_counter(), float(mhz), int(why)))
                except Exception:
                    pass
                time.sleep(0.002)

        self.thread = threading.Thread(target=poll, daemon=True)
        self.thread.start()

    def mark_begin(self):
        self.t_begin = time.perf_counter()

    def mark_end(self):
        self.t_end = time.perf_counter()

    def stop(self):
        self.stop_flag.set()
        if self.thread:
            self.thread.join(1.0)
        rows = self.rows
        if self.t_begin is not None and self.t_end is not None:
            inside = [r for r in rows if self.t_begin <= r[0] <= self.t_end]
            rows = inside or rows
        sm = [r[1] for r in rows]
        reasons = sorted({name for r in rows for bit, name in self.REASONS.items() if r[2] & bit})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(sm), "source": "NVML, polled every 2 ms inside the timed region"}


def step_outputs(ids, obs, est):
    """What a caller of the single-sequence path holds after a step: the feature message the tracker published (ids; x, y,
    z, u, v, vx, vy per feature) and the estimator's window after processImage (p, q wxyz, v, ba, bg per frame; td)."""
    states, td = est.states()
    return {"feature_ids": np.asarray(ids, np.float64), "feature_obs": np.asarray(obs, np.float64),
            "window_states": np.asarray(states, np.float64), "window_td": np.array([td], np.float64)}


def dump_outputs(directory, arrays):
    """--dump-outputs: one float64 .npy file per array, for output-by-output comparison of two builds."""
    os.makedirs(directory, exist_ok=True)
    for name, arr in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), np.asarray(arr, np.float64))


def check_steps(done, wanted, what):
    if done != wanted:
        raise RuntimeError(f"{what}: {done} timed steps instead of the {wanted} asked for (the rendered sequence ran out)")


def make_gpu_pair(device):
    from vins_mono_b200 import FeatureTracker, Estimator
    trk = FeatureTracker(device=device, **synth.tracker_config_dict(**TRK_KW))
    est = Estimator(tic=synth.TIC, ric=synth.RIC, device=device, **EST_KW)
    return trk, est


class TwoStage:
    """Runs a tracker stage (producer thread) and an estimator stage (caller's thread) the way the reference runs its two
    nodes: concurrently, coupled by a bounded queue of feature messages.  The producer stops after `n_before` messages
    until `go()` is called, so that a timed region contains exactly the frames produced after it (pipeline fill and
    drain fall inside the region)."""

    def __init__(self, produce, n_before, n_total, depth=2):
        import queue
        self.q, self.gate, self.err = queue.Queue(maxsize=depth), threading.Event(), None
        self.produce, self.n_before, self.n_total = produce, n_before, n_total
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _run(self):
        try:
            for k in range(self.n_total):
                if k == self.n_before:
                    self.gate.wait()
                msg = self.produce()
                self.q.put(msg)
                if msg is None:
                    return
            self.q.put(None)
        except BaseException as e:  # surfaced by get()
            self.err = e
            self.q.put(None)

    def go(self):
        self.gate.set()

    def get(self):
        msg = self.q.get()
        if self.err:
            raise self.err
        return msg


class SoloGate:
    """Brackets the timed region of ONE sequence: device drained, L2 evicted, optional cross-rank barrier, CUDA events."""

    def __init__(self, device, flush=None, sync_cb=None, clocks=None):
        import torch
        self.torch, self.device, self.flush, self.sync_cb, self.clocks = torch, device, flush, sync_cb, clocks
        self.ev0, self.ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def begin(self):
        if self.flush is not None:
            self.flush.fill_(1.0)
        self.torch.cuda.synchronize(self.device)
        if self.sync_cb:
            self.sync_cb()
        if self.clocks:
            self.clocks.mark_begin()
        self.ev0.record()

    def end(self):
        self.torch.cuda.synchronize(self.device)  # includes the last frame's (asynchronous) marginalisation
        self.ev1.record()
        self.ev1.synchronize()
        if self.clocks:
            self.clocks.mark_end()
        return self.ev0.elapsed_time(self.ev1)


def run_ours_pass(seq, ts, imgs, imu, n_init, warmup, steps, device, host_images, profile=False, flush=None, sync_cb=None,
                  gate=None, d_imgs=None, clocks=None):
    """One pass over the sequence.  The K timed steps form ONE region bracketed by device synchronisation and a pair of
    CUDA events (ms per step = region / K); sync_cb, if given, is the cross-rank barrier placed inside the bracket.
    Tracker and estimator handles are driven from two host threads (TwoStage); with profile=True they run serially."""
    import torch
    trk, est = make_gpu_pair(device)
    if profile:
        trk.set_profile(True)
        est.set_profile(True)
    feeder = BatchedImu(*imu)
    n_pub = n_init + warmup + steps
    est.set_seed(pipeline.gt_seed_rows(seq, ts), seq.ba, seq.bg)
    frame_bytes = imgs.shape[1] * imgs.shape[2]
    if not host_images:
        if d_imgs is None:
            d_imgs = torch.from_numpy(imgs).to(f"cuda:{device}")
        base = d_imgs.data_ptr()
    if gate is None:
        gate = SoloGate(device, flush, sync_cb, clocks)
    launches, h2d, d2h, traj_t, traj_p = 0, 0.0, 0.0, [], []
    n_img = len(ts)
    cursor = [0]

    def one_image(k):
        if host_images:
            return trk.node_image(imgs[k], float(ts[k]))[0]
        return trk.node_image_device(base + k * frame_bytes, imgs.shape[2], float(ts[k]))

    def produce():
        """Images until one publishes -> (stamp, ids, observations, launches, h2d, d2h) or None at end of data."""
        torch.cuda.set_device(device)
        n_l, n_h, n_d, r = 0, 0.0, 0.0, 0
        while r != 2 and cursor[0] < n_img:
            r = one_image(cursor[0])
            cursor[0] += 1
            if r:
                n_l += trk.timing()[1]
                a, b = trk.traffic()
                n_h += a
                n_d += b
        if r != 2:
            return None
        ids, d = pipeline.oracle_feature_message(trk.result())
        return float(ts[cursor[0] - 1]), ids, d, n_l, n_h, n_d

    class Serial:
        def go(self):
            pass

        def get(self):
            return produce()

    stage = Serial() if profile else TwoStage(produce, n_init + warmup, n_pub)
    pubs, first_msg, n_timed, started, last_msg = 0, True, 0, False, None
    while pubs < n_pub:
        timed = pubs >= n_init + warmup
        if timed and not started:
            # start of the timed region: both stages idle, device drained, L2 evicted once (every timed step reads images
            # that were uploaded long ago and never touched since, i.e. cold in L2; the rest of a step's data is
            # produced inside it)
            gate.begin()
            started = True
            stage.go()
        msg = stage.get()
        if msg is None:
            break
        stamp, ids, d, step_launch, step_h2d, step_d2h = msg
        if first_msg:  # estimator_node.cpp:167-172 drops the first feature message
            first_msg = False
        else:
            feeder.feed(est, stamp)
            est.processImage(ids, d, stamp)
            step_launch += est.launch_count()
            a, b = est.traffic()
            step_h2d += a
            step_d2h += b
        if timed:
            n_timed += 1
            launches += step_launch
            h2d += step_h2d
            d2h += step_d2h
            last_msg = (ids, d)
        if est.info()["solver_flag"] == 1:
            st, _ = est.states()
            traj_t.append(stamp)
            traj_p.append(st[-1, 0:3].copy())
        pubs += 1
    region_ms = gate.end() if started else 0.0
    stage.go()
    check_steps(n_timed, steps, "single-sequence pass")
    times = [region_ms / max(n_timed, 1)] * n_timed if started else []
    out = dict(times=times, launches=launches, h2d=h2d, d2h=d2h, traj_t=traj_t, traj_p=traj_p, info=est.info(),
               outputs=step_outputs(*last_msg, est) if last_msg else {})
    if profile:
        out["trk_k"], out["est_k"] = trk.kernel_times(), est.kernel_times()
    trk.close()
    est.close()
    return out


def self_init_check(device, n_pub=80):
    """Untimed: one sequence of geometry-made feature messages through the estimator WITHOUT a seed: the window is bootstrapped by the
    library's own initialStructure (SURVEY 8 next-1).  Reported beside the (seeded) timed runs so that the ATE of a run that owes
    nothing to ground truth is on record."""
    from vins_mono_b200 import Estimator
    try:
        seq = synth.Sequence(seed=0, duration=n_pub / 10.0 + 1.0)
        msgs = synth.track_messages(seq, n_pub, max_feats=150)
        est = Estimator(tic=synth.TIC, ric=synth.RIC, device=device)
        feeder = pipeline.ImuFeeder(*seq.imu())
        tt, pp = [], []
        for k, (stamp, ids, d) in enumerate(msgs):
            if k == 0:
                continue
            feeder.feed(est, stamp)
            est.processImage(ids, d, stamp)
            if est.info()["solver_flag"] == 1:
                st, _ = est.states()
                tt.append(stamp)
                pp.append(st[-1, 0:3].copy())
        ii = est.init_info()
        est.close()
        out = {"self_initialised": ii["self_initialised"], "failed_attempts": ii["failed_attempts"], "reference_frame_l": ii["l"],
               "initial_scale": ii["scale"], "bundle_iterations": ii["bundle_iterations"], "frames_non_linear": len(tt),
               "workload": f"{n_pub} geometry-made feature messages of sequence seed 0 (150 features, 0.3 px noise), 200 Hz IMU, no ve_set_seed"}
        if len(tt) > 25:
            out["ate_rmse_m"] = pipeline.ate_rmse(seq, tt, pp)
            out["ate_rmse_m_after_2s"] = pipeline.ate_rmse(seq, tt, pp, skip=20)
        return out
    except Exception as exc:  # the check must never cost the bench line
        return {"error": repr(exc)}


def distinct_inputs(first_seed, n_distinct, n_pub):
    """Rendered frames + IMU of n_distinct sequences (seeds first_seed ...), enough for n_pub published frames each."""
    return [sequence_inputs(first_seed + d, n_pub) for d in range(n_distinct)]


def run_batch_pass(inputs, n_seq, n_init, warmup, steps, device, host_images=False, flush=None, sync_cb=None, profile=False,
                   clocks=None):
    """n_seq sequences on one GPU through the batched path (vt_batch / ve_batch / vr_open_batch): member k runs the
    distinct sequence k % len(inputs).  One tracker loop and one estimator loop for all members, one launch chain per
    step.  The timed region is ONE vr_advance call of `steps` published frames per member."""
    import torch
    from vins_mono_b200 import TrackerBatch, EstimatorBatch, ReplaySession
    tb = TrackerBatch(n_seq, device=device, **synth.tracker_config_dict(**TRK_KW))
    eb = EstimatorBatch(n_seq, tic=synth.TIC, ric=synth.RIC, device=device, **EST_KW)
    if profile:
        tb.set_profile(True)
        eb.set_profile(True)
    keep, seqs = [], []
    dev_imgs = {}
    for k in range(n_seq):
        d = k % len(inputs)
        seq, ts, imgs, (t_imu, acc, gyr) = inputs[d]
        eb.members[k].set_seed(pipeline.gt_seed_rows(seq, ts), seq.ba, seq.bg)
        if host_images:
            images = dict(images=imgs)
        else:
            if d not in dev_imgs:
                dev_imgs[d] = torch.from_numpy(np.array(imgs, copy=True)).to(f"cuda:{device}")
            images = dict(images=dev_imgs[d].data_ptr(), shape=imgs.shape)
        seqs.append(dict(stamps=ts, imu_t=t_imu, acc=acc, gyr=gyr, **images))
    ses = ReplaySession(tb, eb, seqs)
    gate = SoloGate(device, flush, sync_cb, clocks)
    ses.advance(n_init + warmup)
    before = [ses.stats(k) for k in range(n_seq)]
    gate.begin()
    frames = ses.advance(steps)
    region_ms = gate.end()
    check_steps(frames, steps * n_seq, f"batched pass ({n_seq} sequences x {steps} steps)")
    after = [ses.stats(k) for k in range(n_seq)]
    trajs = [ses.trajectory(k) for k in range(n_seq)]
    infos = [m.info() for m in eb.members]
    windows = [m.states() for m in eb.members]
    outputs = {"window_states": np.stack([w[0] for w in windows]), "window_td": np.array([w[1] for w in windows], np.float64)}
    out = dict(frames=frames, region_ms=region_ms, fps=frames / (region_ms / 1e3) if region_ms else 0.0,
               launches=sum(a_["launches"] - b_["launches"] for a_, b_ in zip(after, before)),
               h2d=sum(a_["h2d"] - b_["h2d"] for a_, b_ in zip(after, before)),
               d2h=sum(a_["d2h"] - b_["d2h"] for a_, b_ in zip(after, before)), trajs=trajs, infos=infos, outputs=outputs)
    out["est_groups"] = eb.groups()
    if profile:
        out["trk_k"], out["est_k"] = tb.kernel_times(), eb.kernel_times()
    ses.close()
    tb.close()
    eb.close()
    del dev_imgs
    return out


def _cv2_tracker_class():
    """The cv2-backed twin of FeatureTracker::readImage + img_callback that generated tests/golden/frontend_track.npz
    (BASELINE.md 3.1: the reference's front end = OpenCV's own kernels); None when cv2 is not importable."""
    try:
        spec = importlib.util.spec_from_file_location("make_frontend_golden", os.path.join(ROOT, "tests", "golden", "make_frontend_golden.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        import cv2
        cv2.setNumThreads(1)        # the reference's tracker node is single threaded
        cv2.setUseOptimized(True)   # the library at its real speed (the golden vectors use the baseline mode for bit-reproducibility)
        return mod.Cv2Tracker
    except Exception:
        return None


def run_reference_pass(seq, ts, imgs, imu, n_init, warmup, steps, front="cv2"):
    """The reference's CPU path on two host threads coupled by a queue like its two nodes (each hot loop single-threaded:
    the tracker node is, and Ceres runs with num_threads = 1).  front = "cv2": OpenCV's own CLAHE / LK / goodFeaturesToTrack /
    findFundamentalMat behind the Python twin of readImage; "port": the oracle's scalar C++ restatement.  Back end: the oracle
    estimator (oracle/, CPU restatement of Estimator + the Ceres dogleg/DENSE_SCHUR loop, tridiagonal-QL eigen-solver)."""
    import orc
    cv2_cls = _cv2_tracker_class() if front == "cv2" else None
    if cv2_cls is not None:
        trk = cv2_cls(synth.tracker_config_dict(**TRK_KW))
        node_image = lambda img, t: trk.node_image(np.ascontiguousarray(img), t)  # noqa: E731
        used = "cv2"
    else:
        trk = orc.OracleTracker(synth.tracker_config_dict(**TRK_KW))
        node_image = lambda img, t: trk.node_image(img, t)[0]  # noqa: E731
        used = "port"
    est = orc.OracleEstimator(orc.be_config(**ORC_KW))
    est.set_fast_eigen(True)  # tridiagonal QL (the reference's Eigen solver class) instead of the parity tests' Jacobi
    feeder = pipeline.ImuFeeder(*imu)
    est.set_seed(pipeline.gt_seed_rows(seq, ts), seq.ba, seq.bg)
    n_pub = n_init + warmup + steps
    traj_t, traj_p = [], []
    cursor = [0]
    t_front = [0.0]

    def produce():
        r = 0
        t0 = time.perf_counter()
        while r != 2 and cursor[0] < len(ts):
            r = node_image(imgs[cursor[0]], float(ts[cursor[0]]))
            cursor[0] += 1
        t_front[0] += time.perf_counter() - t0
        if r != 2:
            return None
        ids, d = pipeline.oracle_feature_message(trk.result())
        return float(ts[cursor[0] - 1]), ids, d

    stage = TwoStage(produce, n_init + warmup, n_pub)
    pubs, first_msg, n_timed, t0, last_msg = 0, True, 0, None, None
    t_back = 0.0
    while pubs < n_pub:
        if pubs == n_init + warmup:
            t0 = time.perf_counter()
            t_front[0] = 0.0
            stage.go()
        msg = stage.get()
        if msg is None:
            break
        stamp, ids, d = msg
        tb0 = time.perf_counter()
        if first_msg:
            first_msg = False
        else:
            feeder.feed(est, stamp)
            est.processImage(ids, d, stamp)
        if t0 is not None:
            n_timed += 1
            t_back += time.perf_counter() - tb0
            last_msg = (ids, d)
        if est.info()["solver_flag"] == 1:
            st, _ = est.states()
            traj_t.append(stamp)
            traj_p.append(st[-1, 0:3].copy())
        pubs += 1
    total_ms = (time.perf_counter() - t0) * 1e3 if t0 is not None else 0.0
    stage.go()
    check_steps(n_timed, steps, "reference pass")
    return dict(times=[total_ms / max(n_timed, 1)] * n_timed, traj_t=traj_t, traj_p=traj_p, front=used,
                front_ms_per_frame=1e3 * t_front[0] / max(n_timed, 1), back_ms_per_frame=1e3 * t_back / max(n_timed, 1),
                outputs=step_outputs(*last_msg, est) if last_msg else {})


def _reference_worker(args):
    seed, n_init, warmup, steps, front = args
    seq, ts, imgs, imu = sequence_inputs(seed, n_init + warmup + steps)
    r = run_reference_pass(seq, ts, imgs, imu, n_init, warmup, steps, front)
    return dict(n=len(r["times"]), total_s=sum(r["times"]) / 1e3, front=r["front"], front_ms=r["front_ms_per_frame"],
                back_ms=r["back_ms_per_frame"], ate=pipeline.ate_rmse(seq, r["traj_t"], r["traj_p"]) if len(r["traj_t"]) > 3 else None)


def run_reference_parallel(seeds, n_init, warmup, steps, front):
    """One CPU pipeline (2 threads) per sequence, as many at a time as the host has core pairs; frames/s = all frames over the
    wall time of the whole pool."""
    import multiprocessing as mp
    procs = max(1, min(len(seeds), (os.cpu_count() or 2) // 2))
    for sd in seeds:  # render (or load from the cache) before forking the workers
        sequence_inputs(sd, n_init + warmup + steps)
    t0 = time.perf_counter()
    with mp.get_context("fork").Pool(procs) as pool:
        res = pool.map(_reference_worker, [(sd, n_init, warmup, steps, front) for sd in seeds], chunksize=1)
    wall = time.perf_counter() - t0
    return res, wall, procs


def _oracle_traj_worker(args):
    """Full CPU oracle pipeline (tracker + estimator twins, Jacobi eigen-solver: the parity configuration) on one sequence."""
    seed, n_pub = args
    import orc
    seq, ts, imgs, imu = sequence_inputs(seed, n_pub)
    trk, est = orc.OracleTracker(synth.tracker_config_dict(**TRK_KW)), orc.OracleEstimator(orc.be_config(**ORC_KW))
    r = pipeline.run_vio(seq, trk, est, len(ts), messages=list(pipeline.feature_messages(trk, ts, imgs))[:n_pub])
    return np.asarray(r["t"]), np.asarray(r["P"])


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def kernel_table(trk_k, est_k):
    kt = {}
    for name, (ms, cnt) in list(trk_k.items()) + list(est_k.items()):
        if cnt:
            kt[name] = {"total_ms": ms, "launches": cnt, "avg_us": 1e3 * ms / cnt}
    return kt


def roofline_object(kt, n_solves, n_images, units_per_launch, peak, peaks_found, note, ba_units_per_launch=None):
    """Dominant kernel by accumulated device time of a profile pass.  Algorithmic bytes per launch = SURVEY 8(d)'s per-unit
    figure (per image for front-end kernels, per solve for BA kernels) x units one launch serves / launches per unit."""
    fe = ("clahe", "pyrdown", "lk_track", "mask_discs", "min_eig", "gftt_tail")
    per_kernel = {}
    for k, v in kt.items():
        if k in fe:
            algo = ALGO_BYTES_IMAGE * n_images * units_per_launch / v["launches"]
        else:
            algo = ALGO_BYTES_SOLVE * n_solves * (ba_units_per_launch or units_per_launch) / v["launches"]
        per_kernel[k] = dict(v, algorithmic_bytes_per_launch=algo, achieved_gbs=algo / (v["avg_us"] * 1e-6) / 1e9,
                             frac=algo / (v["avg_us"] * 1e-6) / 1e9 / peak)
    dominant = max(kt, key=lambda k: kt[k]["total_ms"])
    traffic = None
    try:  # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full captures
        key = dominant if units_per_launch == 1 else f"{dominant}@{units_per_launch}"  # batch captures are stored as name@members
        traffic = json.load(open(os.path.join(ROOT, "profiles", "dram_traffic.json"))).get(key, {}).get("dram_bytes_per_launch")
    except (OSError, ValueError):
        pass
    dk = per_kernel[dominant]
    return {"bound": "hbm", "kernel": dominant, "achieved": dk["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": dk["frac"],
            "traffic": traffic,
            "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst copy)" if peaks_found else "fallback 6650 GB/s",
            "algorithmic_bytes_per_launch": dk["algorithmic_bytes_per_launch"], "avg_launch_us": dk["avg_us"],
            "profiled_solves": n_solves, "profiled_images": n_images, "sequences_per_launch": units_per_launch,
            "note": note, "kernels": per_kernel}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="auto", choices=["auto", "c2", "c3", "c4"],
                    help="auto: configs[1] on one GPU (with a c3 object), configs[4]'s share (64 sequences per GPU) under torchrun")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-frames", type=int, default=150,
                    help="published frames of the CPU-baseline sample inside the b200 arm (~10 s of CPU work)")
    ap.add_argument("--seqs-per-gpu", type=int, default=SEQS_PER_GPU, help="members of the batched workload (configs[2]/[4])")
    ap.add_argument("--distinct", type=int, default=16, help="distinct rendered sequences behind the batch members")
    ap.add_argument("--no-c3", action="store_true", help="skip the configs[2] object of the single-GPU line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed path returned in its last step as DIR/<name>.npy (float64): for one sequence the "
                         "feature message and the estimator window, for a batch every member's window (rank 0's members)")
    a = ap.parse_args()
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    warmup = max(a.warmup, 3) if a.impl == "b200" else a.warmup
    global INIT_PUBS, WORKLOAD
    if a.config == "c4":  # BASELINE configs[3]
        TRK_KW.update(max_cnt=300, min_dist=20)
        EST_KW.update(window_size=20, estimate_td=1, tr=0.033, row=480.0, max_features=2000)
        ORC_KW.update(window_size=20, estimate_td=1, tr=0.033, row=480.0)
        INIT_PUBS, WORKLOAD = 22, WORKLOAD_C4
        a.no_c3 = True
    batched = a.config == "c3" or (a.config == "auto" and world > 1)
    if a.dump_outputs and a.impl == "reference" and batched:
        ap.error("--dump-outputs: the reference arm writes outputs of the single-sequence workload only")
    S = a.seqs_per_gpu
    n_distinct = max(1, min(a.distinct, S))

    if a.impl == "reference":
        if rank != 0:
            return
        front = "cv2" if _cv2_tracker_class() is not None else "port"
        if not batched:
            seq, ts, imgs, imu = sequence_inputs(0, INIT_PUBS + warmup + a.steps)
            r = run_reference_pass(seq, ts, imgs, imu, INIT_PUBS, warmup, a.steps, front)
            if a.dump_outputs:
                dump_outputs(a.dump_outputs, r["outputs"])
            total_s, n = sum(r["times"]) / 1e3, len(r["times"])
            fps, cores = n / total_s, 2
            sample = (f"{n} published frames (2 images + 1 window solve each) of sequence seed 0 after {INIT_PUBS} init + {warmup} "
                      f"warm-up frames")
            extra = {"front_ms_per_frame": r["front_ms_per_frame"], "back_ms_per_frame": r["back_ms_per_frame"]}
            workload, spg = WORKLOAD, 1
            ate = pipeline.ate_rmse(seq, r["traj_t"], r["traj_p"]) if len(r["traj_t"]) > 3 else None
        else:
            # the batched workload on the host: as many sequences at a time as there are core pairs, each a bounded sample
            n_seq_total = S * max(a.gpus, 1)
            procs_cap = max(1, (os.cpu_count() or 2) // 2)
            seeds = list(range(min(n_seq_total, procs_cap, n_distinct * max(a.gpus, 1))))
            steps = a.steps
            res, wall, procs = run_reference_parallel(seeds, INIT_PUBS, warmup, steps, front)
            n = sum(x["n"] for x in res)
            # the pool's wall time contains start-up and the untimed init frames: use the slowest worker's timed region
            total_s = max(x["total_s"] for x in res)
            fps, cores = n / total_s, 2 * procs
            sample = (f"{len(seeds)} of the {n_seq_total} sequences concurrently ({procs} processes x 2 threads on {os.cpu_count()} "
                      f"host cores), {steps} published frames each after {INIT_PUBS} init + {warmup} warm-up frames; aggregate = all "
                      f"frames / slowest pipeline's timed region")
            extra = {"front_ms_per_frame": float(np.mean([x["front_ms"] for x in res])),
                     "back_ms_per_frame": float(np.mean([x["back_ms"] for x in res])), "pool_wall_s": wall}
            workload, spg = WORKLOAD_BATCH.format(s=S, d=n_distinct), S
            ates = [x["ate"] for x in res if x["ate"] is not None]
            ate = float(np.mean(ates)) if ates else None
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": a.gpus, "steps": a.steps,
            "warmup": warmup, "ms_per_step": 1e3 / fps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload, "sequences_per_gpu": spg,
                       "arm": "the same workload on the host CPU: per sequence one tracker thread + one estimator thread"},
            "cpu_baseline": dict({"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample, "cpu": cpu_model(),
                                  "front_end": "OpenCV " + __import__("cv2").__version__ + " (cv2 wheel) behind the Python twin of readImage, 1 thread"
                                  if front == "cv2" else "oracle/ scalar C++ restatement of the OpenCV routines (cv2 not importable)",
                                  "back_end": "oracle/ CPU restatement of Estimator + Ceres dogleg/DENSE_SCHUR (not Ceres itself), own "
                                              "tridiagonal-QL eigen-solver, no wall-clock solver cap"}, **extra),
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "ate_rmse_m": ate,
        }))
        return

    # stdout carries exactly ONE line (the JSON): everything libraries print while the GPUs are set up (NCCL's version banner,
    # torchrun notices) is sent to stderr, stdout is restored for the final print
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(obj), flush=True)

    from vins_mono_b200 import shard
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))

    # frames are rendered (fork pool) before this process touches CUDA; the CPU-baseline sample needs a longer sequence
    cpu_frames = max(a.steps, a.cpu_frames) if (not a.no_cpu_baseline and world == 1 and not batched) else a.steps
    want_c3 = (batched or not a.no_c3)
    c3_steps = a.steps
    batch_inputs = None
    if want_c3:
        first_seed = 100 + shard.sequences_of_rank(rank, world, S)[0]
        batch_inputs = distinct_inputs(first_seed, n_distinct, INIT_PUBS + warmup + c3_steps)
    if not batched:
        seq, ts, imgs, imu = sequence_inputs(shard.sequences_of_rank(rank, world, 1)[0], INIT_PUBS + warmup + cpu_frames)
    # the oracle trajectories of the distinct batch sequences (parity of every member), computed before CUDA exists
    oracle_traj = None
    if want_c3 and rank == 0 and not a.no_cpu_baseline:
        import multiprocessing as mp
        with mp.get_context("fork").Pool(min(n_distinct, max(1, (os.cpu_count() or 2) - 2))) as pool:
            oracle_traj = pool.map(_oracle_traj_worker, [(100 + shard.sequences_of_rank(rank, world, S)[0] + d, INIT_PUBS + warmup + c3_steps)
                                                          for d in range(n_distinct)], chunksize=1)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the vinsb200 library has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"  # keeps NCCL's version banner off stdout: rank 0 prints ONE JSON line
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=f"cuda:{local}")  # 256 MB > 126 MB L2

    def barrier():
        torch.cuda.synchronize(local)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(local)

    rank_barrier = (lambda: dist.barrier()) if world > 1 else None

    def batch_object(with_profile):
        """configs[2] on this GPU: device-resident pass (value), host-image pass (e2e), optional profile pass + parity."""
        run_batch_pass(batch_inputs, min(S, 4), INIT_PUBS, 0, 2, local)  # shake-out
        barrier()
        clk_b = ClockSampler(local)
        clk_b.start()
        rb = run_batch_pass(batch_inputs, S, INIT_PUBS, warmup, c3_steps, local, host_images=False, flush=flush, sync_cb=rank_barrier,
                            clocks=clk_b)
        barrier()
        clocks_b = clk_b.stop()
        barrier()
        re_ = run_batch_pass(batch_inputs, S, INIT_PUBS, warmup, c3_steps, local, host_images=True, flush=flush, sync_cb=rank_barrier)
        barrier()
        obj = {"sequences_per_gpu": S, "distinct_sequences": n_distinct, "frames": rb["frames"], "ms_region": rb["region_ms"],
               "h2d_bytes_per_step": re_["h2d"] / max(re_["frames"], 1), "d2h_bytes_per_step": re_["d2h"] / max(re_["frames"], 1),
               "gpu_launches": rb["launches"], "clocks": clocks_b}
        if with_profile:
            pr = run_batch_pass(batch_inputs, S, INIT_PUBS, 2, min(6, warmup + c3_steps - 2), local, profile=True)
            kt = kernel_table(pr["trk_k"], pr["est_k"])
            n_solves = kt.get("ba_finish", {}).get("launches", 1)
            n_images = kt.get("pyrdown", {}).get("launches", 3) // 3
            obj["roofline"] = roofline_object(kt, n_solves, n_images, S, peak, bool(peaks),
                                              "batched launches: a front-end launch serves all members, a BA launch the members of its launch group "
                                              f"({pr['est_groups']} groups whose chains overlap); algorithmic bytes scale with the members served",
                                              ba_units_per_launch=S / pr["est_groups"])
            obj["estimator_launch_groups"] = pr["est_groups"]
        # parity: every member against the CPU oracle's trajectory of its sequence, and the replicas among themselves
        if oracle_traj is not None:
            worst, worst_rep, n_cmp = 0.0, 0.0, 0
            for k, (tt, pp) in enumerate(rb["trajs"]):
                ot, op = oracle_traj[k % n_distinct]
                m = min(len(tt), len(ot))
                if m and np.array_equal(tt[:m], ot[:m]):
                    worst = max(worst, float(np.abs(pp[:m] - op[:m]).max()))
                    n_cmp += 1
                base = rb["trajs"][k % n_distinct][1]
                mm = min(len(pp), len(base))
                if mm:
                    worst_rep = max(worst_rep, float(np.abs(pp[:mm] - base[:mm]).max()))
            obj["parity"] = {"members_compared": n_cmp, "max_position_dev_vs_oracle_m": worst, "tolerance_m": 3e-4,
                             "ok": bool(n_cmp == len(rb["trajs"]) and worst <= 3e-4), "max_replica_spread_m": worst_rep}
        ates = []
        for k, (tt, pp) in enumerate(rb["trajs"]):
            if len(tt) > 3:
                ates.append(pipeline.ate_rmse(batch_inputs[k % n_distinct][0], tt, pp))
        obj["ate_rmse_m_mean"] = float(np.mean(ates)) if ates else None
        return rb, re_, obj

    if batched:
        rb, re_, obj = batch_object(with_profile=(rank == 0))
        if a.dump_outputs and rank == 0:
            dump_outputs(a.dump_outputs, rb["outputs"])
        fps_dev, t_dev, n_frames = shard.aggregate_rate(rb["region_ms"], rb["frames"], device=f"cuda:{local}")
        fps_e2e, t_e2e, _ = shard.aggregate_rate(re_["region_ms"], re_["frames"], device=f"cuda:{local}")
        launches = torch.tensor([float(rb["launches"])], device=f"cuda:{local}")
        if world > 1:
            dist.all_reduce(launches)
        if rank == 0:
            emit(({
                "impl": "b200", "metric": METRIC, "value": fps_dev, "unit": "frames/s", "n_gpus": world, "steps": c3_steps, "warmup": warmup,
                "ms_per_step": 1e3 * t_dev / c3_steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic",
                "config": {"workload": WORKLOAD_BATCH.format(s=S, d=n_distinct), "sequences_per_gpu": S, "sequences_total": S * world,
                           "step": f"one step = one published frame of every sequence ({S * world} frames); ms_per_step is the time of such a step",
                           "pipelining": "one tracker-batch host thread and one estimator-batch host thread coupled by a depth-2 queue",
                           "l2": "L2 flushed (256 MB write) at the start of the timed region; a step reads 2 x 64 frames (46 MB) that were never touched since upload",
                           "timing": "one CUDA-event pair around the K steps, device synchronised (and ranks barriered) on both sides; max over ranks",
                           "seeded_from_ground_truth": True},
                "e2e": {"value": fps_e2e, "unit": "frames/s", "ms_per_step": 1e3 * t_e2e / c3_steps,
                        "h2d_bytes_per_step": obj["h2d_bytes_per_step"] * S * world, "d2h_bytes_per_step": obj["d2h_bytes_per_step"] * S * world},
                "gpu_launches": int(launches.item()), "roofline": obj.get("roofline"), "cpu_baseline": None, "clocks": obj["clocks"],
                "parity": obj.get("parity"), "ate_rmse_m": obj["ate_rmse_m_mean"],
            }))
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- configs[1]: one sequence ------------------------------------------------------------------------------------
    # untimed shake-out pass (first CUDA context / module load, pinned allocations)
    run_ours_pass(seq, ts, imgs, imu, INIT_PUBS, 0, 2, local, host_images=True)
    clocks = ClockSampler(local)
    barrier()
    clocks.start()
    res_dev = run_ours_pass(seq, ts, imgs, imu, INIT_PUBS, warmup, a.steps, local, host_images=False, flush=flush, sync_cb=rank_barrier,
                            clocks=clocks)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, res_dev["outputs"])
    barrier()
    clk = clocks.stop()
    barrier()
    res_e2e = run_ours_pass(seq, ts, imgs, imu, INIT_PUBS, warmup, a.steps, local, host_images=True, flush=flush, sync_cb=rank_barrier)
    barrier()

    def agg(res):
        rate, sec, _ = shard.aggregate_rate(sum(res["times"]), len(res["times"]), device=f"cuda:{local}")
        return rate, sec

    fps_dev, t_dev = agg(res_dev)
    fps_e2e, t_e2e = agg(res_e2e)

    # ---- roofline of the dominant kernel, measured live with CUDA events in a profile pass
    # 2 warm-up + 10 profiled steps, fewer when the rendered sequence (sized for the timed passes) holds less
    prof = run_ours_pass(seq, ts, imgs, imu, INIT_PUBS, 2, min(10, warmup + cpu_frames - 2), local, host_images=False, profile=True)
    kt = kernel_table(prof["trk_k"], prof["est_k"])
    n_solves = kt.get("ba_finish", {}).get("launches", 1)       # one double2vector launch per solve
    n_images = kt.get("pyrdown", {}).get("launches", 3) // 3      # three pyramid levels per image
    roofline = roofline_object(kt, n_solves, n_images, 1, peak, bool(peaks),
                               "single-sequence step: every kernel is latency/launch bound, not HBM bound (see DESIGN.md)")

    # ---- configs[2]: 64 sequences on this GPU through the batched path
    c3 = None
    if want_c3:
        rb, re_, c3 = batch_object(with_profile=True)
        c3.update({"value": rb["fps"], "unit": "frames/s", "e2e_value": re_["fps"], "steps": c3_steps,
                   "vs_single_sequence": rb["fps"] / fps_dev if fps_dev else None,
                   "note": "BASELINE configs[2]: device-resident frames for value, host frames for e2e_value; one tracker-batch and one "
                           "estimator-batch host thread; same timing bracket as the headline"})

    # ---- CPU baseline on this box's host cores (bounded sample of the same workload)
    cpu_b = None
    ate_ref = ate_same = None
    if not a.no_cpu_baseline:
        rr = run_reference_pass(seq, ts, imgs, imu, INIT_PUBS, warmup, cpu_frames, "cv2")
        tot = sum(rr["times"]) / 1e3
        cpu_b = {"value": len(rr["times"]) / tot, "unit": "frames/s", "cores": 2, "kind": "port", "cpu": cpu_model(),
                 "front_end": rr["front"], "front_ms_per_frame": rr["front_ms_per_frame"], "back_ms_per_frame": rr["back_ms_per_frame"],
                 "sample": f"{len(rr['times'])} published frames of the same sequence after the same {INIT_PUBS} init + {warmup} "
                           f"warm-up frames (front end: {'OpenCV (cv2) twin of readImage' if rr['front'] == 'cv2' else 'oracle scalar port'}, "
                           f"back end: oracle estimator; two threads, {tot:.1f} s)"}
        if rr["front"] == "cv2":  # the all-port figure beside it (scalar C++ tracker), shorter sample
            rp = run_reference_pass(seq, ts, imgs, imu, INIT_PUBS, warmup, min(cpu_frames, 60), "port")
            cpu_b["port_front_end_value"] = len(rp["times"]) / (sum(rp["times"]) / 1e3)
            cpu_b["port_front_ms_per_frame"] = rp["front_ms_per_frame"]
            # trajectories are compared against the port: its tracker is bit-identical to the GPU tracker
            rr_cmp = rp
        else:
            rr_cmp = rr
        nn = min(len(rr_cmp["traj_t"]), len(res_dev["traj_t"]))
        if nn > 3:  # the same frames of both trajectories, so that the two ATE figures are comparable
            ate_ref = pipeline.ate_rmse(seq, rr_cmp["traj_t"][:nn], rr_cmp["traj_p"][:nn])
            ate_same = pipeline.ate_rmse(seq, res_dev["traj_t"][:nn], res_dev["traj_p"][:nn])
    ate = pipeline.ate_rmse(seq, res_dev["traj_t"], res_dev["traj_p"]) if len(res_dev["traj_t"]) > 3 else None

    k = len(res_dev["times"])
    emit(({
        "impl": "b200", "metric": METRIC, "value": fps_dev, "unit": "frames/s", "n_gpus": world, "steps": k, "warmup": warmup,
        "ms_per_step": 1e3 * t_dev / k, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "sequences_per_gpu": 1,
                   "pipelining": "tracker and estimator handles driven from two host threads coupled by a depth-2 queue (the "
                                 "reference's two nodes); the timed region starts with both idle and ends with both drained",
                   "l2": "L2 flushed (256 MB write) at the start of the timed region; every step reads two images that were never touched since upload",
                   "timing": "one CUDA-event pair around the K steps, device synchronised (and ranks barriered) on both sides; max over ranks",
                   "seeded_from_ground_truth": True},
        "e2e": {"value": fps_e2e, "unit": "frames/s", "ms_per_step": 1e3 * t_e2e / k,
                "h2d_bytes_per_step": res_e2e["h2d"] / k, "d2h_bytes_per_step": res_e2e["d2h"] / k},
        "gpu_launches": int(res_dev["launches"]),
        "roofline": roofline, "cpu_baseline": cpu_b, "clocks": clk, "c3": c3,
        "ate_rmse_m": ate, "ate_rmse_m_same_frames": ate_same, "ate_rmse_m_cpu_port": ate_ref,
        "ate_rel_diff": (abs(ate_same - ate_ref) / ate_ref) if ate_ref else None,
        "solver": res_dev["info"], "self_init": self_init_check(local) if rank == 0 else None,
    }))


if __name__ == "__main__":
    main()
