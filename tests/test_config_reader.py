"""vins_mono_b200/config.py: the reference's OpenCV-FileStorage YAML files -> tracker / estimator configurations
(feature_tracker/src/parameters.cpp:37-74, vins_estimator/src/parameters.cpp:42-137).  CPU only."""
import glob
import os

import numpy as np
import pytest

from vins_mono_b200 import config

EUROC_LIKE = """%YAML:1.0

#common parameters
imu_topic: "/imu0"
image_topic: "/cam0/image_raw"
output_path: "/home/tony-ws1/output/"

#camera calibration
model_type: PINHOLE
camera_name: camera
image_width: 752
image_height: 480
distortion_parameters:
   k1: -2.917e-01
   k2: 8.228e-02
   p1: 5.333e-05
   p2: -1.578e-04
projection_parameters:
   fx: 4.616e+02
   fy: 4.603e+02
   cx: 3.630e+02
   cy: 2.481e+02

estimate_extrinsic: 0
extrinsicRotation: !!opencv-matrix
   rows: 3
   cols: 3
   dt: d
   data: [0.0148655429818, -0.999880929698, 0.00414029679422,
           0.999557249008, 0.0149672133247, 0.025715529948,
           -0.0257744366974, 0.00375618835797, 0.999660727178]
extrinsicTranslation: !!opencv-matrix
   rows: 3
   cols: 1
   dt: d
   data: [-0.0216401454975,-0.064676986768, 0.00981073058949]

#feature traker paprameters
max_cnt: 150
min_dist: 30
freq: 10
F_threshold: 1.0
show_track: 1
equalize: 1
fisheye: 0

#optimization parameters
max_solver_time: 0.04
max_num_iterations: 8
keyframe_parallax: 10.0

#imu parameters
acc_n: 0.08
gyr_n: 0.004
acc_w: 0.00004
gyr_w: 2.0e-6
g_norm: 9.81007

estimate_td: 0
td: 0.0
rolling_shutter: 0
rolling_shutter_tr: 0
"""


def test_euroc_style_file():
    from harness import synth
    cfg = config.loads(EUROC_LIKE)
    t, e = config.tracker_kwargs(cfg), config.estimator_kwargs(cfg)
    assert (t["rows"], t["cols"], t["max_cnt"], t["min_dist"], t["freq"], t["equalize"], t["fisheye"], t["camera_model"]) == (480, 752, 150, 30, 10, 1, 0, 0)
    assert (t["fx"], t["fy"], t["cx"], t["cy"], t["k1"], t["p2"]) == (461.6, 460.3, 363.0, 248.1, -0.2917, -1.578e-04) and t["f_threshold"] == 1.0
    assert e["num_iterations"] == 8 and e["estimate_extrinsic"] == 0 and e["estimate_td"] == 0 and e["tr"] == 0.0 and e["row"] == 480.0
    assert (e["acc_n"], e["gyr_n"], e["acc_w"], e["gyr_w"], e["g_norm"], e["keyframe_parallax"]) == (0.08, 0.004, 0.00004, 2.0e-6, 9.81007, 10.0)
    assert np.abs(e["ric"] - synth.RIC).max() < 1e-9 and np.array_equal(e["tic"], synth.TIC)
    assert np.abs(e["ric"] @ e["ric"].T - np.eye(3)).max() < 1e-14     # normalised through a quaternion like the reference
    assert config.ignored(cfg)["max_solver_time"] == 0.04


def test_variants():
    cfg = config.loads(EUROC_LIKE.replace("estimate_extrinsic: 0", "estimate_extrinsic: 2").replace("freq: 10", "freq: 0")
                       .replace("rolling_shutter: 0", "rolling_shutter: 1").replace("rolling_shutter_tr: 0", "rolling_shutter_tr: 0.033")
                       .replace("estimate_td: 0", "estimate_td: 1").replace("td: 0.0", "td: -0.02"))
    e, t = config.estimator_kwargs(cfg), config.tracker_kwargs(cfg)
    assert e["estimate_extrinsic"] == 2 and np.array_equal(e["ric"], np.eye(3)) and np.array_equal(e["tic"], np.zeros(3))
    assert e["tr"] == 0.033 and e["estimate_td"] == 1 and e["td"] == -0.02 and t["freq"] == 100
    mei = config.loads(EUROC_LIKE.replace("model_type: PINHOLE", "model_type: MEI\nmirror_parameters:\n   xi: 2.057")
                       .replace("fx:", "gamma1:").replace("fy:", "gamma2:").replace("cx:", "u0:").replace("cy:", "v0:"))
    t = config.tracker_kwargs(mei)
    assert t["camera_model"] == 1 and t["xi"] == 2.057 and t["fx"] == 461.6 and t["cy"] == 248.1
    with pytest.raises(ValueError):
        config.tracker_kwargs(config.loads(EUROC_LIKE.replace("fisheye: 0", "fisheye: 1")))
    with pytest.raises(ValueError):
        config.tracker_kwargs(config.loads(EUROC_LIKE.replace("model_type: PINHOLE", "model_type: SCARAMUZZA")))


def test_every_configuration_file_of_the_reference_parses():
    # tests/golden/config holds verbatim copies of every config/*/*.yaml file the reference ships
    files = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "config", "*", "*.yaml")))
    assert len(files) == 9
    models = set()
    for f in files:
        cfg = config.load(f)
        e = config.estimator_kwargs(cfg)
        assert e["g_norm"] > 9 and e["num_iterations"] >= 1
        if "image_height" in cfg:  # config/simulation feeds feature messages directly and has no camera section
            mask = np.full((int(cfg["image_height"]), int(cfg["image_width"])), 255, np.uint8) if int(cfg.get("fisheye", 0)) else None
            t = config.tracker_kwargs(cfg, fisheye_mask=mask)
            models.add(t["camera_model"])
            assert t["rows"] > 0 and t["cols"] > 0 and t["fx"] > 0
        assert np.abs(e["ric"] @ e["ric"].T - np.eye(3)).max() < 1e-12
    assert models == {0, 1, 2}      # PINHOLE, MEI and KANNALA_BRANDT configurations all exist in the reference
