"""ORACLE — TEST INFRASTRUCTURE ONLY. ctypes wrapper over oracle/_build/liboracle_exposure.so: auto exposure with light adaptation
(oracle_exposure.cpp, pinned against the reference's own GetWeightedLogLum / UpdateAverageLuminancePS), and `AutoExposureChain`, the
oracle chain of oracle_py.Oracle with the measured, adapted luminance in place of the constant ave_log_lum - what the product chain
computes with dfx_chain_config.auto_exposure set.

Importers: tests/ and tools/. Never the product path.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(_HERE, "_build", "liboracle_exposure.so")
SOURCES = ["oracle_exposure.cpp"]
HEADERS = ["oracle_exposure.h", "oracle_common.h", "oracle_math.h", "oracle_tex.h", "oracle_quant.h"]
# the flags of oracle/Makefile: scalar C++, no FMA contraction
CXXFLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fvisibility=hidden", "-Wall", "-Wextra", "-Wno-unused-parameter", "-pthread"]
H01 = float(np.float16(0.1))  # the R16F state cleared to 0.1 (EpipolarLightScattering.cpp:885-905)


def build(force: bool = False) -> str:
    deps = [os.path.join(_HERE, f) for f in SOURCES + HEADERS]
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(f) for f in deps):
        os.makedirs(os.path.dirname(LIB), exist_ok=True)
        tmp = LIB + f".{os.getpid()}.tmp"
        subprocess.check_call([os.environ.get("CXX", "g++"), *CXXFLAGS, "-shared", "-o", tmp, *[os.path.join(_HERE, f) for f in SOURCES]])
        os.replace(tmp, LIB)
    return LIB


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(LIB)
        for f in ("orc_weighted_log_lum", "orc_update_average_luminance_ps"):
            getattr(L, f).restype = None
        _lib = L
    return _lib


def _fp(a: np.ndarray):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def weighted_log_lum(rgb: np.ndarray) -> np.ndarray:
    """GetWeightedLogLum (AtmosphereShadersCommon.fxh:199-205, MinLuminance 0.01) per row of an (..., 3) array -> (..., 2)."""
    a = np.ascontiguousarray(rgb, np.float32).reshape(-1, 3)
    out = np.empty((a.shape[0], 2), np.float32)
    lib().orc_weighted_log_lum(_fp(a), _fp(out), a.shape[0])
    return out.reshape(np.asarray(rgb).shape[:-1] + (2,))


def update_average_luminance_ps(loglum_w: np.ndarray, elapsed, light_adaptation: bool) -> np.ndarray:
    """UpdateAverageLuminancePS (UpdateAverageLuminance.fx:12-29) per row of an (N, 2) array of (wlogL, w) -> (N, 2) (exp(LogLum), weight)."""
    a = np.ascontiguousarray(loglum_w, np.float32).reshape(-1, 2)
    dt = np.ascontiguousarray(np.broadcast_to(np.asarray(elapsed, np.float32), (a.shape[0],)))
    out = np.empty_like(a)
    lib().orc_update_average_luminance_ps(_fp(a), _fp(dt), int(bool(light_adaptation)), _fp(out), a.shape[0])
    return out


def update_average_luminance(rgba: np.ndarray, sampling: int, elapsed: float, light_adaptation: bool, state=None) -> np.ndarray:
    """One auto-exposure update of `state` (value, max(0.05, value), measurement, weight; default: the cleared state) from an
    (H, W, 4) frame: sampling 1 = the reference's 64x64 point samples and half-rounded mip chain, 2 = every pixel, fp64 sum."""
    a = np.ascontiguousarray(rgba, np.float32)
    st = np.array([H01, H01, 0.0, 0.0] if state is None else state, np.float32)
    r = lib().orc_update_average_luminance(_fp(a), a.shape[1], a.shape[0], int(sampling), C.c_float(elapsed), int(bool(light_adaptation)), _fp(st))
    if r != 0:
        raise ValueError("bad arguments to orc_update_average_luminance")
    return st


class AutoExposureChain:
    """oracle_py.Oracle's whole-frame sequence with auto exposure, as the product chain runs it with dfx_chain_config.auto_exposure =
    `mode` (1 = reference sampling, 2 = every pixel): when the tone-map attribs have bAutoExposure set, the plane Bloom receives is
    measured before the composite, the state adapts over `elapsed` seconds per frame (bLightAdaptation), and ToneMap() uses
    max(0.05, state). The state restarts at 0.1 whenever the frame indices are not consecutive (the chain's history reset rule)."""

    def __init__(self, oracle, mode: int, elapsed: float = 0.0):
        from diligentfx_b200.capi import ToneMapAttribs
        self.o, self.mode, self.elapsed = oracle, int(mode), float(elapsed)
        self.set_tonemap(ToneMapAttribs.default(), 0.3, True)
        self.state = np.array([H01, H01, 0.0, 0.0], np.float32)
        self.frame_index, self.last = 0, None

    def set_tonemap(self, a, ave_log_lum: float = 0.3, to_srgb: bool = True):
        self.tm, self.ave_log_lum, self.to_srgb = a, float(ave_log_lum), bool(to_srgb)
        self.o.set_tonemap(a, ave_log_lum, to_srgb)

    def set_inputs(self, fr: dict):
        self.o.set_inputs(fr)
        self.frame_index = int(fr["frame"])

    def average_luminance(self) -> np.ndarray:
        """(state, max(0.05, state), this frame's measurement, its blend weight) after the last frame()."""
        return self.state.copy()

    def frame(self, stages: int = 127) -> None:
        o, idx = self.o, self.frame_index
        exposure = self.mode != 0 and self.tm.bAutoExposure != 0 and bool(stages & 64)
        if not exposure:
            o.frame(stages)
        else:
            o.frame(stages & ~64)
            if self.last is None or idx != self.last + 1:
                self.state = np.array([H01, H01, 0.0, 0.0], np.float32)
            bloom = bool(stages & 32)
            self.state = update_average_luminance(o.get("bloom_in") if bloom else o.get("color"), self.mode, self.elapsed,
                                                  self.tm.bLightAdaptation != 0, self.state)
            o.set("tonemap_in", o.get("bloom_out") if bloom else o.get("color"))
            o.set_tonemap(self.tm, float(self.state[1]), self.to_srgb)
            o.run("tonemap")
            o.set_tonemap(self.tm, self.ave_log_lum, self.to_srgb)
        self.last = idx

    def get(self, name: str) -> np.ndarray:
        return self.o.get(name)
