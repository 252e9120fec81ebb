"""Auto exposure with light adaptation on the device (csrc/dfx_exposure.cu): the luminance measurement and its adaptation state
against the CPU oracle (oracle/oracle_exposure.cpp, oracle/exposure_py.py), the tone-map entries that read the state from device memory, and the chain
with dfx_chain_config.auto_exposure (eager == graph replay, overlap == one stream, fused == unfused, streaming == frame by frame)."""
import ctypes as C

import numpy as np
import pytest

from helpers import Dev, psnr, rows
from diligentfx_b200 import capi, synth
from oracle import exposure_py as op
from oracle import oracle_py

pytestmark = pytest.mark.gpu

REF, FULL = capi.LUMINANCE_SAMPLING_REFERENCE, capi.LUMINANCE_SAMPLING_FULL
H01 = float(np.float16(0.1))


def _state(d: Dev):
    t = d.empty(1, capi.AVERAGE_LUMINANCE_STATE_FLOATS, 1)
    capi.check(d.lib.dfx_pass_reset_average_luminance(None, C.c_void_p(t.data_ptr())), "reset")
    return t


def _update(d: Dev, state, color_t, sampling, dt, adapt=True):
    a = capi.ToneMapAttribs.default()
    a.bLightAdaptation = int(adapt)
    p = d.plane(color_t)
    capi.check(d.lib.dfx_pass_update_average_luminance(None, C.byref(a), sampling, C.c_float(dt), C.byref(p), C.c_void_p(state.data_ptr())), "update")


def _hdr_frames(w, h, n, seed=11):
    """A synthetic HDR sequence whose exposure changes: the chain's colour scaled by a per-frame factor, plus a moving highlight."""
    rng = np.random.default_rng(seed)
    base = synth.noise_frame(w, h, seed)["color"].astype(np.float32)
    out = []
    for k in range(n):
        c = base * np.float32(0.2 * 2.0 ** (k % 5))
        y0, x0 = (k * 7) % max(h - 4, 1), (k * 13) % max(w - 4, 1)
        c[y0:y0 + 3, x0:x0 + 3, :3] = np.float32(50.0)
        c[..., 3] = 1.0
        c[rng.random((h, w)) < 0.05, :3] = 0.0  # black pixels: weight 0
        out.append(np.ascontiguousarray(c))
    return out


def test_reference_mode_matches_oracle_bit_for_bit():
    d = Dev()
    w, h = 333, 187
    dts = [0.0, 0.016, 0.1, 0.5, 0.033, 2.0, 0.008, 1.0]
    st = _state(d)
    want = np.array([H01, H01, 0, 0], np.float32)
    for k, (c, dt) in enumerate(zip(_hdr_frames(w, h, 8), dts)):
        _update(d, st, d.up(c), REF, dt)
        want = op.update_average_luminance(c, 1, dt, True, want)
        got = Dev.host(st)[0, :4]
        assert got[0] == want[0] and got[1] == want[1], (k, got, want)
        assert got[2] == want[2] and got[3] == want[3], (k, got, want)


def test_reference_mode_reads_rgba16f_like_rgba32f():
    import torch
    d = Dev()
    c = _hdr_frames(96, 54, 1)[0].astype(np.float16)
    s32, s16 = _state(d), _state(d)
    _update(d, s32, d.up(c.astype(np.float32)), REF, 0.0, adapt=False)
    t16 = torch.from_numpy(np.ascontiguousarray(c)).cuda()
    d.keep.append(t16)
    _update(d, s16, t16, REF, 0.0, adapt=False)
    assert np.array_equal(Dev.host(s32)[0, :4], Dev.host(s16)[0, :4])


@pytest.mark.parametrize("w,h", [(1920, 1080), (3840, 2160)])
def test_full_mode_against_fp64_oracle_and_deterministic(w, h):
    d = Dev()
    c = _hdr_frames(w, h, 1, seed=3)[0]
    ct = d.up(c)
    s1, s2 = _state(d), _state(d)
    _update(d, s1, ct, FULL, 0.0, adapt=False)
    _update(d, s2, ct, FULL, 0.0, adapt=False)
    a, b = Dev.host(s1)[0], Dev.host(s2)[0]
    assert np.array_equal(a[:4], b[:4])
    want = op.update_average_luminance(c, 2, 0.0, False)
    rel = abs(float(a[2]) - float(want[2])) / float(want[2])
    assert rel <= 1e-5, (a[:4], want)
    # a second launch on the same buffer starts from a clean ticket and blends onto the first result
    _update(d, s1, ct, FULL, 0.5, adapt=True)
    assert Dev.host(s1)[0, 2] == a[2]


@pytest.mark.parametrize("mode", list(range(12)))
@pytest.mark.parametrize("x", [0.01, 0.37])
def test_dev_tonemap_entries_equal_scalar_entries(mode, x):
    d = Dev()
    w, h = 96, 54
    rng = np.random.default_rng(mode)
    color = d.up(np.abs(rng.normal(0.5, 1.0, (h, w, 4))).astype(np.float32))
    up0 = d.up(np.abs(rng.normal(0.3, 0.5, (h // 2, w // 2, 4))).astype(np.float32))
    st = d.up(np.array([x, max(0.05, x)] + [0.0] * 6, np.float32))
    tm = capi.ToneMapAttribs.default()
    tm.iToneMappingMode = mode
    bl = capi.BloomAttribs.default()
    L = d.lib
    o_s, o_d, f_s, f_d = (d.empty(h, w, 4) for _ in range(4))
    P = d.plane
    for srgb in (0, 1):
        capi.check(L.dfx_pass_tonemap(None, C.byref(tm), C.c_float(max(0.05, x)), srgb, C.byref(P(color)), C.byref(P(o_s)), rows(h)))
        capi.check(L.dfx_pass_tonemap_dev(None, C.byref(tm), C.c_void_p(st.data_ptr()), srgb, C.byref(P(color)), C.byref(P(o_d)), rows(h)))
        capi.check(L.dfx_pass_bloom_composite_tonemap(None, C.byref(bl), C.byref(tm), C.c_float(max(0.05, x)), srgb, C.byref(P(color)), C.byref(P(up0)),
                                                      C.byref(P(f_s)), rows(h)))
        capi.check(L.dfx_pass_bloom_composite_tonemap_dev(None, C.byref(bl), C.byref(tm), C.c_void_p(st.data_ptr()), srgb, C.byref(P(color)),
                                                          C.byref(P(up0)), C.byref(P(f_d)), rows(h)))
        assert np.array_equal(Dev.host(o_s), Dev.host(o_d))
        assert np.array_equal(Dev.host(f_s), Dev.host(f_d))


# ---------------------------------------------------------------------------------------------------------------------------------
# chain
# ---------------------------------------------------------------------------------------------------------------------------------
W, H, N = 192, 108, 7
DTS = [0.016, 0.05, 0.3, 0.016, 1.0, 0.1, 0.02]


@pytest.fixture(scope="module")
def seq():
    s = synth.generate_sequence(W, H, N)
    for k, fr in enumerate(s):  # exposure changes over the sequence
        fr["color"] = np.ascontiguousarray(fr["color"] * np.float32(2.0 ** (k % 3 - 1)))
    return s


def _run(seq, frames=None, **kw):
    import torch
    from diligentfx_b200.chain import ChainConfig, PostProcessChain
    ch = PostProcessChain(W, H, ChainConfig(**kw))
    outs, states = [], []
    for k, fr in enumerate(seq if frames is None else frames):
        ch.upload(fr)
        ldr = ch.execute(fr["frame"], fr["curr_camera"], fr["prev_camera"], elapsed_time=DTS[k % len(DTS)])
        torch.cuda.synchronize()
        outs.append(ldr.cpu().numpy().copy())
        states.append(ch.average_luminance())
    stats = ch.stats()
    ch.close()
    return outs, states, stats


@pytest.mark.parametrize("ae", [1, 2])
def test_chain_eager_graph_overlap_fused_agree(seq, ae):
    base, st0, stats0 = _run(seq, auto_exposure=ae, graph=False, overlap=False, fuse=False)
    assert stats0["frames_replayed"] == 0
    for kw in (dict(graph=True, overlap=True, fuse=True), dict(graph=True, overlap=False, fuse=True), dict(graph=False, overlap=True, fuse=False),
               dict(graph=True, overlap=True, fuse=False)):
        outs, st, stats = _run(seq, auto_exposure=ae, **kw)
        if kw["graph"]:
            assert stats["frames_replayed"] > 0, stats
        for k in range(N):
            assert np.array_equal(outs[k], base[k]), (kw, k)
            assert st[k] == st0[k], (kw, k)
    # the exposure actually moves: the state is not the cleared value after a few frames
    assert st0[-1]["state"] != H01


def test_chain_auto_exposure_off_by_attribs_equals_constant(seq):
    from diligentfx_b200.capi import ToneMapAttribs
    tm = ToneMapAttribs.default()
    tm.bAutoExposure = 0
    a, _, _ = _run(seq, auto_exposure=1, tonemap=tm)
    b, _, _ = _run(seq, auto_exposure=0)
    for k in range(N):
        assert np.array_equal(a[k], b[k])


def test_chain_streaming_equals_frame_by_frame(seq):
    import torch
    from diligentfx_b200.chain import ChainConfig, PostProcessChain
    want, _, _ = _run(seq, auto_exposure=2)
    ch = PostProcessChain(W, H, ChainConfig(auto_exposure=2))
    frames = [dict(fr, elapsed_time=DTS[k % len(DTS)]) for k, fr in enumerate(seq)]
    res = [torch.empty((H, W, 4), dtype=torch.float32).pin_memory() for _ in range(N)]
    ch.stream_frames(frames, ldr_host=res)
    torch.cuda.synchronize()
    for k in range(N):
        assert np.array_equal(res[k].numpy(), want[k]), k
    ch.close()


def test_chain_history_reset_restarts_state(seq):
    import torch
    from diligentfx_b200.chain import ChainConfig, PostProcessChain
    ch = PostProcessChain(W, H, ChainConfig(auto_exposure=1))
    ch.set_elapsed_time(1e6)  # weight 1: the state is the measurement
    for fr in seq[:3]:
        ch.run_frame(fr)
    s = ch.average_luminance()
    assert s["weight"] == 1.0 and s["state"] == float(np.float16(s["measured"]))
    # a frame index that does not follow: histories reset, the luminance restarts from 0.1 before this frame's update
    ch.set_elapsed_time(0.0)
    fr = dict(seq[0], frame=100)
    ch.upload(fr)
    ch.execute(100, fr["curr_camera"], fr["prev_camera"])
    torch.cuda.synchronize()
    assert ch.average_luminance()["state"] == H01
    ch.close()


def test_chain_4k_against_oracle_chain():
    import torch
    from diligentfx_b200.chain import ChainConfig, PostProcessChain
    w, h = 3840, 2160
    s = synth.generate_sequence(w, h, 2)
    for ae in (1, 2):
        ch = PostProcessChain(w, h, ChainConfig(auto_exposure=ae))
        o = op.AutoExposureChain(oracle_py.Oracle(w, h), ae, 0.05)
        for fr in s:
            ch.upload(fr)
            ldr = ch.execute(fr["frame"], fr["curr_camera"], fr["prev_camera"], elapsed_time=0.05)
            o.set_inputs(fr)
            o.frame()
        torch.cuda.synchronize()
        got = np.clip(ldr.cpu().numpy()[..., :3], 0, 1)
        want = np.clip(o.get("ldr")[..., :3], 0, 1)
        assert psnr(got, want) >= 49.0
        gs, ws = ch.average_luminance(), o.average_luminance()
        assert abs(gs["measured"] - ws[2]) <= 1e-3 * ws[2], (gs, ws)
        assert abs(gs["state"] - ws[0]) <= 1e-3 * ws[0], (gs, ws)
        ch.close()
