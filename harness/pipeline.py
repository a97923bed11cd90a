"""ROS-free replay driver: rendered sequence -> feature tracker -> estimator, the way the reference's two nodes
exchange data (feature_tracker_node.cpp:113-165 packs, estimator_node.cpp:98-136, 209-339 aligns IMU with the
feature message and calls processIMU / processImage).  Works with any tracker / estimator objects exposing
node_image()/feature_message() and processIMU()/processImage()/states() — the CUDA product or the CPU oracle."""
from __future__ import annotations

import hashlib
import os
import tempfile

import numpy as np

from . import synth


def cached_images(seq: synth.Sequence, n: int, cache_dir=None):
    """The first n rendered images of seq, cached as .npy in a per-user directory under the system's temporary directory
    (never in the source tree, which may be read-only).  A file appears under its final name only once it is complete, so
    concurrent processes never read a partial one; a cache that cannot be written only costs the next call a render."""
    if cache_dir is None:
        cache_dir = os.path.join(tempfile.gettempdir(), f"vinsb200_cache-{os.getuid()}")
    key = hashlib.sha1(f"{seq.seed}-{seq.rows}x{seq.cols}-{seq.pixel_noise}-{seq.cam_hz}-{n}-v2".encode()).hexdigest()[:16]
    path = os.path.join(cache_dir, key + ".npy")
    ts = seq.image_times()[:n]
    if os.path.exists(path):
        return ts, np.load(path, mmap_mode="r")
    _, imgs = seq.images(n)
    tmp = None
    try:
        os.makedirs(cache_dir, mode=0o700, exist_ok=True)
        fd, tmp = tempfile.mkstemp(dir=cache_dir, suffix=".partial")
        with os.fdopen(fd, "wb") as f:
            np.save(f, imgs)
        os.replace(tmp, path)
    except OSError:
        if tmp is not None and os.path.exists(tmp):
            os.unlink(tmp)
    return ts, imgs


def oracle_feature_message(res):
    """PointCloud payload from a tracker result dict (track_cnt > 1 only)."""
    keep = res["track_cnt"] > 1
    ids = res["ids"][keep]
    un, cur, vel = res["un_pts"][keep], res["cur_pts"][keep], res["velocity"][keep]
    d = np.zeros((len(ids), 7))
    d[:, 0:2], d[:, 2], d[:, 3:5], d[:, 5:7] = un, 1.0, cur, vel
    return ids.astype(np.int32), d


def feature_messages(tracker, ts, imgs):
    """Yields (stamp, ids, xyz_uv_vel[n,7]) for every published frame (img_callback semantics)."""
    for i in range(len(ts)):
        r, _ = tracker.node_image(np.ascontiguousarray(imgs[i]), float(ts[i]))
        if r == 2:
            yield float(ts[i]), *oracle_feature_message(tracker.result())


def gt_seed_rows(seq: synth.Sequence, stamps):
    rows = []
    for t in stamps:
        p, R, v, _, _ = seq.pose(t)
        rows.append(np.r_[t, p, synth.rot_to_quat_wxyz(R), v])
    return np.array(rows)


class ImuFeeder:
    """estimator_node.cpp:98-136 (getMeasurements) + :225-265 (per-sample dt, interpolation at the image stamp)."""

    def __init__(self, t, acc, gyr):
        self.t, self.acc, self.gyr = t, acc, gyr
        self.k = 0
        self.current_time = -1.0

    def feed(self, estimator, stamp, td=None):
        """img_t = stamp + estimator.td, both for the sample selection and for the interpolation at the image
        (estimator_node.cpp:106-126, 232-265); td defaults to the estimator's current estimate."""
        if td is None:
            td = estimator.states()[1] if hasattr(estimator, "states") else 0.0
        img_t = stamp + td
        n = len(self.t)
        while self.k < n and self.t[self.k] < img_t:
            self._one(estimator, self.k, img_t)
            self.k += 1
        if self.k < n:  # the first sample at/after the image stamp is used but stays in the buffer
            self._one(estimator, self.k, img_t)

    def _one(self, estimator, k, img_t):
        t = self.t[k]
        if t <= img_t:
            if self.current_time < 0:
                self.current_time = t
            dt = t - self.current_time
            self.current_time = t
            self._d = (self.acc[k].copy(), self.gyr[k].copy())
            estimator.processIMU(dt, self.acc[k], self.gyr[k])
        else:
            dt_1, dt_2 = img_t - self.current_time, t - img_t
            self.current_time = img_t
            w1, w2 = dt_2 / (dt_1 + dt_2), dt_1 / (dt_1 + dt_2)
            a = w1 * self._d[0] + w2 * self.acc[k]
            g = w1 * self._d[1] + w2 * self.gyr[k]
            self._d = (a, g)
            estimator.processIMU(dt_1, a, g)


def run_vio(seq: synth.Sequence, tracker, estimator, n_images, messages=None, on_frame=None):
    """Returns dict(t, P[n,3], Q[n,4] wxyz of the newest window frame after each processImage once NON_LINEAR)."""
    t_imu, acc, gyr = seq.imu()
    feeder = ImuFeeder(t_imu, acc, gyr)
    if messages is None:
        ts, imgs = cached_images(seq, n_images)
        messages = list(feature_messages(tracker, ts, imgs))
    all_stamps = [m[0] for m in messages]
    estimator.set_seed(gt_seed_rows(seq, all_stamps), seq.ba, seq.bg)
    out_t, out_P, out_Q = [], [], []
    first = True
    for stamp, ids, d in messages:
        if first:  # estimator_node.cpp:167-172 drops the first feature message
            first = False
            continue
        feeder.feed(estimator, stamp)
        estimator.processImage(ids, d, stamp)
        info = estimator.info()
        if info["solver_flag"] == 1:
            st, _ = estimator.states()
            out_t.append(stamp)
            out_P.append(st[-1, 0:3].copy())
            out_Q.append(st[-1, 3:7].copy())
        if on_frame:
            on_frame(stamp, estimator)
    return dict(t=np.array(out_t), P=np.array(out_P), Q=np.array(out_Q), messages=messages)


def ate_rmse(seq: synth.Sequence, t, P, skip=0):
    """RMSE absolute trajectory error after an SE(3) (rotation + translation, no scale) Umeyama alignment."""
    t, P = np.asarray(t)[skip:], np.asarray(P)[skip:]
    G = np.array([seq.pose(ti)[0] for ti in t])
    mu_p, mu_g = P.mean(0), G.mean(0)
    H = (P - mu_p).T @ (G - mu_g)
    U, _, Vt = np.linalg.svd(H)
    D = np.diag([1, 1, np.sign(np.linalg.det(Vt.T @ U.T))])
    R = Vt.T @ D @ U.T
    aligned = (R @ (P - mu_p).T).T + mu_g
    return float(np.sqrt(np.mean(np.sum((aligned - G) ** 2, axis=1))))
