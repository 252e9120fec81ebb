"""REFERENCE-SHADER RUNNER — TEST INFRASTRUCTURE ONLY. The reference's auto-exposure shaders (EpipolarLightScattering's
GetWeightedLogLum and UpdateAverageLuminancePS, LIGHT_ADAPTATION 0 and 1) behind harness/exposure.inc, compiled for the CPU exactly as
build_ref.py compiles the PostProcess passes (same rewrites, same flags, shader text read in place, never written into the repository)
into a library of their own, oracle/_ref/librefexposure.so.

    python oracle/refshader/build_exposure.py [--force]
"""
from __future__ import annotations

import ctypes as C
import importlib.util
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(os.path.dirname(HERE), "_ref", "librefexposure.so")


def _build_ref():
    spec = importlib.util.spec_from_file_location("dfx_refshader_build", os.path.join(HERE, "build_ref.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def passes() -> list[dict]:
    # EpipolarLightScattering.cpp:1799-1802: LIGHT_ADAPTATION = bLightAdaptation, LOW_RES_LUMINANCE_MIPS = 7 (64x64);
    # ShaderUtilities.fxh names the HLSL `matrix` type
    return [{"name": f"exposure__adapt{la}", "shader": "UpdateAverageLuminance.fx", "harness": "exposure.inc",
             "macros": {"SUPPORTED_SHADER_SRV": 1, "LIGHT_ADAPTATION": la, "LOW_RES_LUMINANCE_MIPS": 7, "matrix": "float4x4"}} for la in (0, 1)]


def available() -> bool:
    return os.path.exists(LIB)


def build(force: bool = False) -> str:
    """Builds where the reference is mounted; elsewhere a library that exists is used as is."""
    br = _build_ref()
    if not os.path.isdir(br.REF_SHADERS):
        return LIB
    os.makedirs(os.path.join(br.OUT_DIR, "obj"), exist_ok=True)
    idx = br._index()
    objs = []
    for p in passes():
        name, obj, err = br._compile(p, idx, force)
        if err:
            raise RuntimeError(f"{name}: compile failed\n{err[:6000]}")
        objs.append(obj)
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(o) for o in objs):
        subprocess.check_call(["g++", "-shared", "-pthread", "-o", LIB, *objs])
    return LIB


_lib = None


def run(name: str, ins, outs, iparams=(), threads: int = 0) -> None:
    """One full-screen pass of `name` (exposure__adapt0 / exposure__adapt1), the calling convention of refsh.run."""
    global _lib
    sys.path.insert(0, HERE)
    import refsh
    if _lib is None:
        _lib = C.CDLL(LIB)
    ins = [np.ascontiguousarray(a, np.float32) for a in ins]
    pin = (refsh.Plane * max(len(ins), 1))(*[refsh._plane(a) for a in ins])
    pout = (refsh.Plane * max(len(outs), 1))(*[refsh._plane(a) for a in outs])
    ip = (C.c_int * max(len(iparams), 1))(*[int(v) for v in iparams])
    cb_ptr, cb_size = (C.c_void_p * 1)(), (C.c_int * 1)()
    a = refsh.Args(pin, len(ins), pout, len(outs), cb_ptr, cb_size, 0, ip, len(iparams), None, threads or (os.cpu_count() or 1))
    fn = getattr(_lib, "refsh_" + name)
    fn.restype = C.c_int
    r = fn(C.byref(a))
    if r != 0:
        raise RuntimeError(f"refsh_{name} failed with {r}")


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
