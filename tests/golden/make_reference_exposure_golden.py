"""Writes tests/golden/reference_exposure_record.npz: inputs and outputs of the reference's own auto-exposure shaders
(GetWeightedLogLum, UpdateAverageLuminancePS with LIGHT_ADAPTATION 0 and 1), run through oracle/_ref/librefexposure.so
(oracle/refshader/build_exposure.py), so that
tests/test_auto_exposure_cpu.py compares the oracle with them where the shader library cannot be built.

    python tests/golden/make_reference_exposure_golden.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "tests", "golden", "reference_exposure_record.npz")
H, W = 27, 49


def inputs():
    rng = np.random.default_rng(20261017)
    color = np.zeros((H, W, 4), np.float32)
    color[..., :3] = np.exp2(rng.uniform(-12, 8, (H, W, 3)))
    color[0] = 0.0                                       # black: weight 0
    color[1, :, :3] = np.float32(0.01)                   # at the luminance threshold
    color[2, :, :3] = np.float32(0.02)                   # weight 1
    color[..., 3] = 1.0
    lw = np.zeros((H, W, 4), np.float32)
    lw[..., 0] = rng.normal(-1.0, 2.5, (H, W))
    lw[..., 1] = rng.choice([0.0, 1e-7, 5e-4, 1e-3, 0.25, 1.0], (H, W))
    dt = np.zeros((H, W, 4), np.float32)
    dt[..., 0] = rng.choice([0.0, 1.0 / 60, 0.1, 0.5, 3.0], (H, W))
    return color, lw, dt


def run_reference(color, lw, dt):
    from oracle.refshader import build_exposure as refsh
    wll = np.zeros((H, W, 2), np.float32)
    refsh.run("exposure__adapt0", [color], [wll], iparams=[0])
    upd = []
    for la in (0, 1):
        o = np.zeros((H, W, 4), np.float32)
        refsh.run(f"exposure__adapt{la}", [lw, dt], [o], iparams=[1])
        upd.append(o)
    return wll, upd[0], upd[1]


if __name__ == "__main__":
    c, lw, dt = inputs()
    wll, u0, u1 = run_reference(c, lw, dt)
    np.savez_compressed(OUT, color=c, loglum_w=lw, elapsed=dt, weighted_log_lum=wll, update_adapt0=u0, update_adapt1=u1)
    print("wrote", OUT)
