"""ctypes view of include/dfx_b200.h (the C-ABI of libdfx_b200.so).

Only structure layouts, the library loader and small plane helpers live here; all arithmetic is in the CUDA
library. Loading fails loudly when the library is missing or when a declared symbol is not exported: there is
no Python/CPU fallback for any pass.
"""
from __future__ import annotations

import ctypes as C
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
REPO_ROOT = os.path.dirname(_HERE)
LIB_PATH = os.environ.get("DFX_LIB") or os.path.join(_HERE, "lib", "libdfx_b200.so")  # DFX_LIB: another build of the same library (tuning sweeps)
HEADER_PATH = os.path.join(REPO_ROOT, "include", "dfx_b200.h")

DFX_OK, DFX_ERR_INVALID_ARG, DFX_ERR_CUDA, DFX_ERR_NOT_PREPARED, DFX_ERR_UNSUPPORTED = range(5)
FORMAT_R32F, FORMAT_RG32F, FORMAT_RGBA32F, FORMAT_R8U = 1, 2, 3, 4
FORMAT_RGBA16F, FORMAT_RG16F, FORMAT_RG8U, FORMAT_RGBA8U = 5, 6, 7, 8   # transfer formats (unpack / pack only)
MAX_MIPS = 8

TAA_FLAG_GAUSSIAN, TAA_FLAG_BICUBIC, TAA_FLAG_YCOCG = 1, 2, 4
SSR_FLAG_PREVIOUS_FRAME = 1
POSTFX_FLAG_REVERSED_DEPTH = 1
SSAO_FLAG_HALF_RESOLUTION = 2
SSR_FLAG_HALF_RESOLUTION = 2
# auto exposure (dfx_pass_update_average_luminance, dfx_chain_config.auto_exposure)
AUTO_EXPOSURE_OFF, LUMINANCE_SAMPLING_REFERENCE, LUMINANCE_SAMPLING_FULL = 0, 1, 2
AVERAGE_LUMINANCE_MAX_PARTIALS = 512
AVERAGE_LUMINANCE_STATE_FLOATS = 8 + 2 * AVERAGE_LUMINANCE_MAX_PARTIALS   # [0] state, [1] max(0.05, state), [2] measurement, [3] its weight


class Float4x4(C.Structure):
    _fields_ = [("m", (C.c_float * 4) * 4)]


class CameraAttribs(C.Structure):
    _fields_ = [
        ("f4Position", C.c_float * 4), ("f4ViewportSize", C.c_float * 4),
        ("fNearPlaneZ", C.c_float), ("fFarPlaneZ", C.c_float), ("fNearPlaneDepth", C.c_float), ("fFarPlaneDepth", C.c_float),
        ("fSceneNearZ", C.c_float), ("fSceneFarZ", C.c_float), ("fSceneNearDepth", C.c_float), ("fSceneFarDepth", C.c_float),
        ("fHandness", C.c_float), ("uiFrameIndex", C.c_uint32), ("Padding0", C.c_float), ("Padding1", C.c_float),
        ("fFocusDistance", C.c_float), ("fFStop", C.c_float), ("fFocalLength", C.c_float), ("fSensorWidth", C.c_float),
        ("fSensorHeight", C.c_float), ("fExposure", C.c_float), ("f2Jitter", C.c_float * 2),
        ("mView", Float4x4), ("mProj", Float4x4), ("mViewProj", Float4x4),
        ("mViewInv", Float4x4), ("mProjInv", Float4x4), ("mViewProjInv", Float4x4),
        ("f4ExtraData", (C.c_float * 4) * 5),
    ]


class SSAOAttribs(C.Structure):
    _fields_ = [("EffectRadius", C.c_float), ("EffectFalloffRange", C.c_float), ("RadiusMultiplier", C.c_float),
                ("DepthMIPSamplingOffset", C.c_float), ("TemporalStabilityFactor", C.c_float),
                ("SpatialReconstructionRadius", C.c_float), ("ResetAccumulation", C.c_int32), ("AlphaInterpolation", C.c_float),
                ("BitmaskThickness", C.c_float), ("Algorithm", C.c_uint32), ("Padding0", C.c_float), ("Padding1", C.c_float)]

    @staticmethod
    def default() -> "SSAOAttribs":
        return SSAOAttribs(1.0, 0.615, 1.457, 3.3, 0.9, 4.0, 0, 1.0, 0.5, 0, 0.0, 0.0)


class SSRAttribs(C.Structure):
    _fields_ = [("DepthBufferThickness", C.c_float), ("RoughnessThreshold", C.c_float), ("MostDetailedMip", C.c_uint32),
                ("IsRoughnessPerceptual", C.c_int32), ("RoughnessChannel", C.c_uint32), ("MaxTraversalIntersections", C.c_uint32),
                ("GGXImportanceSampleBias", C.c_float), ("SpatialReconstructionRadius", C.c_float),
                ("TemporalRadianceStabilityFactor", C.c_float), ("TemporalVarianceStabilityFactor", C.c_float),
                ("BilateralCleanupSpatialSigmaFactor", C.c_float), ("AlphaInterpolation", C.c_float)]

    @staticmethod
    def default() -> "SSRAttribs":
        return SSRAttribs(0.025, 0.2, 0, 1, 0, 128, 0.3, 4.0, 1.0, 0.9, 0.9, 1.0)


class BloomAttribs(C.Structure):
    _fields_ = [("Intensity", C.c_float), ("Threshold", C.c_float), ("SoftTreshold", C.c_float), ("Radius", C.c_float),
                ("AlphaInterpolation", C.c_float), ("Padding0", C.c_float), ("Padding1", C.c_float), ("Padding2", C.c_float)]

    @staticmethod
    def default() -> "BloomAttribs":
        return BloomAttribs(0.15, 1.0, 0.125, 0.75, 1.0, 0.0, 0.0, 0.0)


class DOFAttribs(C.Structure):
    _fields_ = [("MaxCircleOfConfusion", C.c_float), ("TemporalStabilityFactor", C.c_float), ("BokehKernelRingCount", C.c_int32),
                ("BokehKernelRingDensity", C.c_int32), ("AlphaInterpolation", C.c_float), ("Padding0", C.c_float), ("Padding1", C.c_float),
                ("Padding2", C.c_float)]

    @staticmethod
    def default() -> "DOFAttribs":
        return DOFAttribs(0.01, 0.9375, 5, 7, 1.0, 0.0, 0.0, 0.0)


DOF_FLAG_TEMPORAL_SMOOTHING, DOF_FLAG_KARIS_INVERSE = 1, 2


class TAAAttribs(C.Structure):
    _fields_ = [("TemporalStabilityFactor", C.c_float), ("ResetAccumulation", C.c_int32), ("SkipRejection", C.c_int32),
                ("Padding0", C.c_float)]

    @staticmethod
    def default() -> "TAAAttribs":
        return TAAAttribs(0.9375, 0, 0, 0.0)


class ToneMapAttribs(C.Structure):
    _fields_ = [("iToneMappingMode", C.c_int32), ("bAutoExposure", C.c_int32), ("fMiddleGray", C.c_float),
                ("bLightAdaptation", C.c_int32), ("fWhitePoint", C.c_float), ("fLuminanceSaturation", C.c_float),
                ("Padding0", C.c_uint32), ("Padding1", C.c_uint32),
                ("AgXSaturation", C.c_float), ("AgXSlope", C.c_float), ("AgXPower", C.c_float), ("AgXOffset", C.c_float)]

    @staticmethod
    def default() -> "ToneMapAttribs":
        return ToneMapAttribs(4, 1, 0.18, 1, 3.0, 1.0, 0, 0, 1.0, 1.0, 1.0, 0.0)


class FrameDesc(C.Structure):
    _fields_ = [("Index", C.c_uint32), ("Width", C.c_uint32), ("Height", C.c_uint32), ("OutputWidth", C.c_uint32),
                ("OutputHeight", C.c_uint32)]


class Plane(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("pitch_bytes", C.c_size_t), ("width", C.c_int32), ("height", C.c_int32),
                ("format", C.c_int32), ("flags", C.c_int32)]


class Pyramid(C.Structure):
    _fields_ = [("level", Plane * MAX_MIPS), ("levels", C.c_int32), ("reserved", C.c_int32)]


class Rows(C.Structure):
    _fields_ = [("y0", C.c_int32), ("y1", C.c_int32)]


MAX_PEERS = 8


class PeerSet(C.Structure):
    """dfx_peer_set (include/dfx_b200.h): base pointers of the row-strip-sharded planes per owning rank."""
    _fields_ = [("count", C.c_int32), ("row_begin", C.c_int32 * (MAX_PEERS + 1)), ("color", C.c_void_p * MAX_PEERS),
                ("normal", C.c_void_p * MAX_PEERS), ("hiz", (C.c_void_p * MAX_PEERS) * MAX_MIPS)]


class PeerMap(C.Structure):
    """dfx_peer_map: slab bases of the ranks sharing a frame + the 64-row aligned strip boundaries."""
    _fields_ = [("count", C.c_int32), ("rank", C.c_int32), ("row_begin", C.c_int32 * (MAX_PEERS + 1)), ("base", C.c_void_p * MAX_PEERS)]


class PostFXRenderAttribs(C.Structure):
    _fields_ = [("stream", C.c_void_p), ("curr_depth", C.POINTER(Plane)), ("prev_depth", C.POINTER(Plane)),
                ("motion_vectors", C.POINTER(Plane)), ("curr_camera", C.POINTER(CameraAttribs)),
                ("prev_camera", C.POINTER(CameraAttribs))]


class SSAORenderAttribs(C.Structure):
    _fields_ = [("stream", C.c_void_p), ("postfx", C.c_void_p), ("depth", C.POINTER(Plane)), ("normal", C.POINTER(Plane)),
                ("attribs", C.POINTER(SSAOAttribs))]


class SSRRenderAttribs(C.Structure):
    _fields_ = [("stream", C.c_void_p), ("postfx", C.c_void_p), ("color", C.POINTER(Plane)), ("depth", C.POINTER(Plane)),
                ("normal", C.POINTER(Plane)), ("material", C.POINTER(Plane)), ("motion", C.POINTER(Plane)),
                ("attribs", C.POINTER(SSRAttribs))]


class BloomRenderAttribs(C.Structure):
    _fields_ = [("stream", C.c_void_p), ("postfx", C.c_void_p), ("color", C.POINTER(Plane)), ("attribs", C.POINTER(BloomAttribs))]


class TAARenderAttribs(C.Structure):
    _fields_ = [("stream", C.c_void_p), ("postfx", C.c_void_p), ("color", C.POINTER(Plane)), ("attribs", C.POINTER(TAAAttribs)),
                ("accumulation_buffer_idx", C.c_uint32)]


class DOFRenderAttribs(C.Structure):
    _fields_ = [("stream", C.c_void_p), ("postfx", C.c_void_p), ("color", C.POINTER(Plane)), ("depth", C.POINTER(Plane)),
                ("attribs", C.POINTER(DOFAttribs))]


assert C.sizeof(DOFAttribs) == 32


class ChainConfigC(C.Structure):
    """dfx_chain_config (include/dfx_b200.h, chain level)."""
    _fields_ = [("ssao", SSAOAttribs), ("ssr", SSRAttribs), ("bloom", BloomAttribs), ("taa", TAAAttribs), ("tonemap", ToneMapAttribs), ("dof", DOFAttribs),
                ("postfx_flags", C.c_uint32), ("ssao_flags", C.c_uint32), ("ssr_flags", C.c_uint32), ("taa_flags", C.c_uint32), ("dof_flags", C.c_uint32),
                ("stages", C.c_uint32), ("enable_dof", C.c_int32), ("fuse", C.c_int32), ("overlap", C.c_int32), ("use_graph", C.c_int32), ("to_srgb", C.c_int32),
                ("ave_log_lum", C.c_float), ("ssr_scale", C.c_float), ("ssao_scale", C.c_float), ("auto_exposure", C.c_int32)]


class ChainFrame(C.Structure):
    """dfx_chain_frame."""
    _fields_ = [("frame_index", C.c_uint32), ("defer_post", C.c_int32), ("curr_camera", C.POINTER(CameraAttribs)), ("prev_camera", C.POINTER(CameraAttribs)),
                ("depth", C.POINTER(Plane)), ("prev_depth", C.POINTER(Plane)), ("motion", C.POINTER(Plane)), ("normal", C.POINTER(Plane)),
                ("color", C.POINTER(Plane)), ("material", C.POINTER(Plane)), ("ldr_out", C.POINTER(Plane))]


class ChainStats(C.Structure):
    _fields_ = [("frames_eager", C.c_uint64), ("frames_replayed", C.c_uint64), ("graphs_built", C.c_uint64), ("graph_failures", C.c_uint64)]


CHAIN_EFFECT = {"postfx": 0, "ssao": 1, "ssr": 2, "bloom": 3, "taa": 4, "dof": 5}
assert C.sizeof(CameraAttribs) == 576 and C.sizeof(SSAOAttribs) == 48 and C.sizeof(SSRAttribs) == 48
assert C.sizeof(BloomAttribs) == 32 and C.sizeof(TAAAttribs) == 16 and C.sizeof(ToneMapAttribs) == 48


def declared_symbols(header_path: str = HEADER_PATH) -> list[str]:
    """Every `DFX_API` function declared in include/dfx_b200.h."""
    text = open(header_path).read()
    return sorted(set(re.findall(r"DFX_API\s+[\w\s\*]+?\b(dfx_\w+)\s*\(", text)))


class DfxError(RuntimeError):
    pass


_lib = None


def load(path: str = LIB_PATH) -> C.CDLL:
    """Load libdfx_b200.so (no compute is triggered; safe without a GPU)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(path):
        raise DfxError(f"{path} is missing: build it first (python -c 'import __graft_entry__ as g; g.build()'). "
                       "There is no CPU fallback.")
    lib = C.CDLL(path)
    lib.dfx_last_error.restype = C.c_char_p
    lib.dfx_launch_count.restype = C.c_uint64
    lib.dfx_postfx_get_camera_attribs_dev.restype = C.c_void_p
    lib.dfx_bloom_mip_count.restype = C.c_int32
    lib.dfx_chain_effect.restype = C.c_void_p
    lib.dfx_chain_post_stream.restype = C.c_void_p
    lib.dfx_chain_average_luminance_dev.restype = C.c_void_p
    lib.dfx_chain_set_elapsed_time.argtypes = [C.c_void_p, C.c_float]
    for name in declared_symbols():
        if not hasattr(lib, name):
            raise DfxError(f"libdfx_b200.so does not export {name}")
    _lib = lib
    return lib


def check(status: int, what: str = "") -> None:
    if status != DFX_OK:
        msg = load().dfx_last_error()
        raise DfxError(f"{what} failed with status {status}: {msg.decode() if msg else ''}")


_FMT_OF = {(1,): FORMAT_R32F, (2,): FORMAT_RG32F, (4,): FORMAT_RGBA32F}


PLANE_FLAG_REVERSED_DEPTH = 1


def plane_of(t, fmt: int | None = None, flags: int = 0) -> Plane:
    """Describe a contiguous torch CUDA tensor (H,W), (H,W,2) or (H,W,4) float32 / (H,W) uint8 as a dfx_plane; transfer
    formats: (H,W,4) / (H,W,2) float16 and (H,W,2) / (H,W,4) uint8."""
    import torch
    assert t.is_cuda and t.is_contiguous(), "plane tensors must be contiguous CUDA tensors"
    h, w = int(t.shape[0]), int(t.shape[1])
    if t.dtype == torch.uint8:
        f, bpp = {2: (FORMAT_R8U, 1), 3: {2: (FORMAT_RG8U, 2), 4: (FORMAT_RGBA8U, 4)}.get(int(t.shape[-1]))}[t.dim()]
    elif t.dtype == torch.float16:
        f, bpp = {2: (FORMAT_RG16F, 4), 4: (FORMAT_RGBA16F, 8)}[int(t.shape[2])]
    else:
        assert t.dtype == torch.float32
        ch = 1 if t.dim() == 2 else int(t.shape[2])
        f, bpp = _FMT_OF[(ch,)], 4 * ch
    if fmt is not None:
        assert fmt == f
    return Plane(t.data_ptr(), w * bpp, w, h, f, flags)


def pyramid_of(tensors, flags: int = 0) -> Pyramid:
    """`flags` go on level 0 (the depth buffer a depth pyramid is built from)."""
    p = Pyramid()
    p.levels = len(tensors)
    for i, t in enumerate(tensors):
        p.level[i] = plane_of(t, flags=flags if i == 0 else 0)
    return p


def rows_all(h: int) -> Rows:
    return Rows(0, h)
