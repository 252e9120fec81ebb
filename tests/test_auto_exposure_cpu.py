"""Auto exposure with light adaptation, CPU side: the oracle's restatement (oracle/oracle_exposure.cpp) against the reference's own
shaders (live through oracle/_ref/librefexposure.so, or against the committed record tests/golden/reference_exposure_record.npz),
known answers of the measurement and the adaptation, and the C-ABI's argument checks (no kernel is launched)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from diligentfx_b200 import capi
from oracle import exposure_py as op

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RECORD = os.path.join(ROOT, "tests", "golden", "reference_exposure_record.npz")
H01 = float(np.float16(0.1))


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


# ---------------------------------------------------------------------------------------------------------------------------------
# oracle == reference shaders
# ---------------------------------------------------------------------------------------------------------------------------------
def _reference_outputs():
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import make_reference_exposure_golden as g
    rec = np.load(RECORD)
    from oracle.refshader import build_exposure
    if build_exposure.available():
        live = g.run_reference(rec["color"], rec["loglum_w"], rec["elapsed"])
        # the record is what the shaders compute today
        for name, a in zip(("weighted_log_lum", "update_adapt0", "update_adapt1"), live):
            assert np.array_equal(_bits(a), _bits(rec[name])), f"{name}: the record is stale (python {g.__file__})"
    return rec


def test_weighted_log_lum_matches_reference_shader():
    rec = _reference_outputs()
    got = op.weighted_log_lum(rec["color"][..., :3])
    assert np.array_equal(_bits(got), _bits(rec["weighted_log_lum"]))


@pytest.mark.parametrize("adapt", [0, 1])
def test_update_average_luminance_ps_matches_reference_shader(adapt):
    rec = _reference_outputs()
    lw, dt = rec["loglum_w"], rec["elapsed"]
    got = op.update_average_luminance_ps(lw[..., :2].reshape(-1, 2), dt[..., 0].reshape(-1), bool(adapt)).reshape(lw.shape[:2] + (2,))
    want = rec[f"update_adapt{adapt}"]
    assert np.array_equal(_bits(got[..., 0]), _bits(want[..., 0]))
    assert np.array_equal(_bits(got[..., 1]), _bits(want[..., 3]))


# ---------------------------------------------------------------------------------------------------------------------------------
# known answers
# ---------------------------------------------------------------------------------------------------------------------------------
def _const(h, w, lum):
    c = np.zeros((h, w, 4), np.float32)
    c[..., :3] = np.float32(lum)  # grey: luminance = lum * (sum of the weights) = lum within an ulp
    c[..., 3] = 1.0
    return c


@pytest.mark.parametrize("sampling", [1, 2])
@pytest.mark.parametrize("lum", [0.02, 0.18, 3.5])
def test_constant_colour_without_adaptation(sampling, lum):
    c = _const(27, 49, lum)
    L = np.float32(lum) * np.float32(0.212671) + np.float32(lum) * np.float32(0.715160) + np.float32(lum) * np.float32(0.072169)
    s = op.update_average_luminance(c, sampling, 0.25, False)
    if sampling == 1:  # every stored value is half: state = half(exp(half(log L)))
        want = np.float16(np.exp(np.float32(np.float16(np.log(np.float32(L))))))
        assert s[0] == np.float32(want), (s, want)
    else:
        assert abs(s[0] - L) <= L * 2.0 ** -10
    assert s[3] == 1.0 and s[1] == max(0.05, s[0])


@pytest.mark.parametrize("sampling", [1, 2])
def test_adaptation_follows_exponential(sampling):
    L, dt = 1.5, 0.2
    c = _const(54, 96, L)
    s = None
    for n in range(1, 25):
        s = op.update_average_luminance(c, sampling, dt, True, s)
        want = L + (0.1 - L) * np.exp(-n * dt)
        assert abs(s[0] - want) <= 2e-3 * max(want, 0.1) * n ** 0.5 + 2.0 ** -10 * L, (n, s[0], want)


@pytest.mark.parametrize("sampling", [1, 2])
def test_black_frame_leaves_state_unchanged(sampling):
    c = _const(27, 49, 0.0)
    c[::3, ::5, :3] = 0.005  # below MinLuminance 0.01: still weight 0
    st = np.array([np.float16(0.73), np.float16(0.73), 0, 0], np.float32)
    s = op.update_average_luminance(c, sampling, 0.5, True, st)
    assert s[0] == st[0] and s[3] == 0.0
    s = op.update_average_luminance(c, sampling, 0.5, False)
    assert s[0] == np.float32(H01)


def test_tone_map_luminance_clamp():
    s = op.update_average_luminance(_const(16, 16, 0.011), 1, 0.0, False)  # luminance just above the threshold: a dark frame
    assert s[0] < 0.05 and s[1] == np.float32(0.05)
    s = op.update_average_luminance(_const(16, 16, 0.5), 1, 0.0, False)
    assert s[1] == s[0] > 0.05


@pytest.mark.parametrize("w,h", [(49, 27), (1920, 1080), (64, 64), (7, 5)])
def test_reference_sample_positions(w, h):
    """The 64x64 samples read texel floor((i + .5) / 64 * size): a frame that is bright exactly there and black elsewhere measures
    the bright value; moving the bright texels by one loses them."""
    xs = np.floor((np.arange(64, dtype=np.float32) + np.float32(0.5)) * np.float32(1 / 64) * np.float32(w)).astype(int)
    ys = np.floor((np.arange(64, dtype=np.float32) + np.float32(0.5)) * np.float32(1 / 64) * np.float32(h)).astype(int)
    c = _const(h, w, 0.0)
    c[np.ix_(ys, xs)] = _const(1, 1, 2.0)[0, 0]
    s = op.update_average_luminance(c, 1, 0.0, False)
    assert abs(s[2] - 2.0) <= 2.0 * 2.0 ** -9
    if w >= 128 and h >= 128:
        c2 = _const(h, w, 0.0)
        c2[np.ix_(ys + 1, xs + 1)] = _const(1, 1, 2.0)[0, 0]
        assert op.update_average_luminance(c2, 1, 0.0, False)[3] == 0.0


def test_oracle_chain_with_auto_exposure():
    """AutoExposureChain: off (mode 0 or bAutoExposure = 0) it is the plain oracle chain; on, it tone-maps with the luminance measured on
    the plane Bloom receives, and a frame index that does not follow restarts the state at 0.1."""
    from diligentfx_b200 import synth
    from oracle import oracle_py
    w, h = 96, 54
    seq = synth.generate_sequence(w, h, 3)

    def run(mode, auto=1, frames=seq):
        ch = op.AutoExposureChain(oracle_py.Oracle(w, h, threads=4), mode, 0.5)
        tm = capi.ToneMapAttribs.default()
        tm.bAutoExposure = auto
        ch.set_tonemap(tm, 0.3, True)
        states = []
        for fr in frames:
            ch.set_inputs(fr)
            ch.frame()
            states.append(ch.average_luminance())
        return ch, states

    plain = oracle_py.Oracle(w, h, threads=4)
    for fr in seq:
        plain.set_inputs(fr)
        plain.frame()
    off, _ = run(1, auto=0)
    assert np.array_equal(off.get("ldr"), plain.get("ldr"))
    on, states = run(1)
    want = None
    for k, fr in enumerate(seq):  # replay the measurement on the oracle's own Bloom input of each frame
        o = oracle_py.Oracle(w, h, threads=4)
        for f in seq[:k + 1]:
            o.set_inputs(f)
            o.frame()
        want = op.update_average_luminance(o.get("bloom_in"), 1, 0.5, True, want)
        assert np.array_equal(states[k], want), k
    assert not np.array_equal(on.get("ldr"), plain.get("ldr"))
    _, reset = run(2, frames=[seq[0], dict(seq[1], frame=10)])
    ref = oracle_py.Oracle(w, h, threads=4)
    ref.set_inputs(dict(seq[1], frame=10))
    ref.frame()
    assert np.array_equal(reset[1], op.update_average_luminance(ref.get("bloom_in"), 2, 0.5, True))  # from the cleared state


# ---------------------------------------------------------------------------------------------------------------------------------
# C-ABI (no kernel launched)
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib(built):
    return capi.load()


def test_symbols_exported(lib):
    for n in ("dfx_pass_update_average_luminance", "dfx_pass_reset_average_luminance", "dfx_pass_tonemap_dev", "dfx_pass_bloom_composite_tonemap_dev",
              "dfx_chain_set_elapsed_time", "dfx_chain_average_luminance_dev"):
        assert n in capi.declared_symbols() and hasattr(lib, n), n


def test_arguments_rejected_before_launch(lib):
    a = capi.ToneMapAttribs.default()
    buf = (C.c_float * capi.AVERAGE_LUMINANCE_STATE_FLOATS)()  # any 16-byte aligned address: validation happens first
    state = C.c_void_p((C.addressof(buf) + 15) & ~15)
    plane = capi.Plane(C.addressof(buf) + 64, 64, 4, 4, capi.FORMAT_RGBA32F, 0)
    upd = lib.dfx_pass_update_average_luminance
    assert upd(None, None, 1, C.c_float(0.0), C.byref(plane), state) == capi.DFX_ERR_INVALID_ARG
    assert upd(None, C.byref(a), 1, C.c_float(0.0), None, state) == capi.DFX_ERR_INVALID_ARG
    assert upd(None, C.byref(a), 1, C.c_float(0.0), C.byref(plane), None) == capi.DFX_ERR_INVALID_ARG
    for bad in (0, 3, -1):
        assert upd(None, C.byref(a), bad, C.c_float(0.0), C.byref(plane), state) == capi.DFX_ERR_INVALID_ARG
    assert upd(None, C.byref(a), 1, C.c_float(-1.0), C.byref(plane), state) == capi.DFX_ERR_INVALID_ARG
    assert upd(None, C.byref(a), 1, C.c_float(0.0), C.byref(plane), C.c_void_p(state.value + 4)) == capi.DFX_ERR_INVALID_ARG
    r16 = capi.Plane(C.addressof(buf) + 64, 16, 4, 4, capi.FORMAT_R32F, 0)
    assert upd(None, C.byref(a), 1, C.c_float(0.0), C.byref(r16), state) == capi.DFX_ERR_INVALID_ARG
    assert lib.dfx_pass_reset_average_luminance(None, None) == capi.DFX_ERR_INVALID_ARG
    assert lib.dfx_pass_tonemap_dev(None, C.byref(a), None, 1, C.byref(plane), C.byref(plane), capi.Rows(0, 4)) == capi.DFX_ERR_INVALID_ARG
    b = capi.BloomAttribs.default()
    assert lib.dfx_pass_bloom_composite_tonemap_dev(None, C.byref(b), C.byref(a), None, 1, C.byref(plane), C.byref(plane), C.byref(plane),
                                                    capi.Rows(0, 4)) == capi.DFX_ERR_INVALID_ARG
    lib.dfx_chain_set_elapsed_time.argtypes = [C.c_void_p, C.c_float]
    assert lib.dfx_chain_set_elapsed_time(None, 0.1) == capi.DFX_ERR_INVALID_ARG
    lib.dfx_chain_average_luminance_dev.restype = C.c_void_p
    assert lib.dfx_chain_average_luminance_dev(None) is None


def test_chain_config_default_auto_exposure_off(lib):
    c = capi.ChainConfigC()
    lib.dfx_chain_config_default(C.byref(c))
    assert c.auto_exposure == 0 and C.sizeof(c) == 284
    assert c.tonemap.bAutoExposure == 1 and c.tonemap.bLightAdaptation == 1  # the reference defaults, ignored unless auto_exposure is set
    from diligentfx_b200.chain import ChainConfig
    assert ChainConfig().auto_exposure == 0


def test_shim_overload_compiles(tmp_path):
    src = r'''
#include "dfx/PostProcessEffects.hpp"
void f(Diligent::IDeviceContext* ctx, Diligent::ITextureView* c, Diligent::ITextureView* o, const Diligent::HLSL::ToneMappingAttribs& tm)
{
    Diligent::AverageLuminance lum(Diligent::AverageLuminance::SAMPLING_REFERENCE);
    lum.Update(ctx, c, tm, 1.0 / 60.0);
    Diligent::ToneMap(ctx, c, o, tm, lum, 0.3f, true);
    Diligent::ToneMap(ctx, c, o, tm, lum.GetStateDev(), true);
    lum.Reset(ctx);
}
'''
    f = tmp_path / "shim_exposure.cpp"
    f.write_text(src)
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(f)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
