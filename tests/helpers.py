"""Shared test helpers: golden fixtures, calibration."""
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_calib_c1():
    d = json.load(open(os.path.join(GOLDEN, "calib_c1.json")))
    return {k: np.array(v, np.float64) for k, v in d.items()}


def scaled_calib(c, sc, sp):
    """Reference calibration scaled to another resolution (SURVEY.md 8d): fx,fy,cx,cy times
    W/1600 (camera) or PW/1280 (projector); distortion and extrinsics unchanged."""
    out = {k: v.copy() for k, v in c.items()}
    for key, s in (("Kc", sc), ("Kp", sp)):
        K = out[key].reshape(3, 3).copy()
        K[0, 0] *= s; K[1, 1] *= s; K[0, 2] *= s; K[1, 2] *= s
        out[key] = K.ravel()
    return out


def load_c1_crop():
    return dict(np.load(os.path.join(GOLDEN, "c1_crop.npz")))


def load_c1_full():
    """The reference's whole captured scan (tools/make_golden.py c1full)."""
    return dict(np.load(os.path.join(GOLDEN, "c1_full.npz")))
