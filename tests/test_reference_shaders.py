"""Pins the oracle against the reference ITSELF: every pass of the oracle is compared with the reference's own HLSL pixel
shader for that pass, compiled for the CPU by oracle/refshader (sources read in place from the reference, never copied) and
run on the same inputs.

Bar: BIT-EXACT. The shader runner and the oracle state the HLSL intrinsics and the fixed-function sampler the same way
(fp32, no contraction, 1/256-texel bilinear snap), so any difference is a difference between the oracle's restatement and
the reference's shader text. The one tolerated pass is the first bokeh gather of DepthOfField, whose 142 bilinear taps per
pixel are aimed with a texture coordinate the shader derives from the interpolated NDC position (0.5 + 0.5 * ndc) while
the oracle uses (x + 0.5) / W: the last-bit difference moves a few taps across a 1/256-texel snap boundary.

Where oracle/_ref/librefshaders.so exists (build() makes it wherever the reference's sources are at hand) the shaders run
live, and tests/golden/reference_shader_record.json must still hold exactly what they produce. Everywhere else the oracle is
compared with that record of the shaders' outputs: a SHA-256 digest of every plane, bit for bit, and for the planes compared
with a tolerance a fixed sample of their texels (tests/golden/reference_shader_samples.npz). To rewrite both after a
deliberate change, where the library exists:

    DFX_RECORD_REFERENCE_SHADERS=1 python -m pytest tests/test_reference_shaders.py
"""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

from diligentfx_b200 import capi, synth
from oracle.refshader import refsh

from oracle.refshader.driver import Variant, compare_frame, make_oracle

W, H = 157, 89                                   # odd on both axes: the odd-size branches of every mip chain run
TOLERATED = {"D8 dof_bokeh_first.near": (1e-3, 0.02), "D8 dof_bokeh_first.far": (1e-3, 0.02)}   # (max abs, max fraction of texels that differ)
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RECORD = os.path.join(GOLDEN, "reference_shader_record.json")
SAMPLES = os.path.join(GOLDEN, "reference_shader_samples.npz")
SAMPLE_TEXELS = 256
RECORDING = bool(os.environ.get("DFX_RECORD_REFERENCE_SHADERS"))
_recorded = {"planes": {}, "constant_buffers": {}, "samples": {}}


@pytest.fixture(scope="module")
def shaders(built):
    """True where the reference's shaders run live, False where the oracle is compared with their recorded outputs."""
    try:
        refsh.build()
    except Exception as e:                       # pragma: no cover - only where the reference is present but does not compile
        pytest.fail(f"the reference shaders no longer compile for the CPU: {e}")
    if RECORDING and not refsh.available():
        pytest.fail("recording the reference shaders' outputs needs oracle/_ref/librefshaders.so")
    yield refsh.available()
    if RECORDING:
        with open(RECORD, "w") as f:
            json.dump({k: _recorded[k] for k in ("planes", "constant_buffers")}, f, indent=1, sort_keys=True)
            f.write("\n")
        np.savez_compressed(SAMPLES, **_recorded["samples"])


_record = None


def _load_record():
    global _record
    if _record is None:
        with open(RECORD) as f:
            _record = json.load(f)
        with np.load(SAMPLES) as z:
            _record["samples"] = {k: z[k] for k in z.files}
    return _record


def _digest(a: np.ndarray) -> str:
    a = np.ascontiguousarray(a, np.float32)
    return hashlib.sha256(repr(a.shape).encode() + a.tobytes()).hexdigest()


def _sample(a: np.ndarray) -> np.ndarray:
    """A fixed, evenly spaced sample of the plane's texels (every channel)."""
    flat = np.ascontiguousarray(a, np.float32).reshape(a.shape[0] * a.shape[1], -1)
    return flat[np.linspace(0, flat.shape[0] - 1, min(SAMPLE_TEXELS, flat.shape[0])).round().astype(np.int64)]


def _run(v: Variant, live: bool, frames=None, warm: int = 2):
    seq = frames if frames is not None else synth.generate_sequence(W, H, warm + 1)
    h, w = seq[0]["depth"].shape
    o = make_oracle(w, h, v)
    o.set_reversed_depth(v.reversed_depth)
    try:
        for fr in seq[:warm]:
            o.set_inputs(fr)
            o.frame(v.stages())
        return compare_frame(o, seq[warm], v, with_reference=live)
    finally:
        o.set_reversed_depth(False)


def _difference(label: str, got: np.ndarray, want: np.ndarray, rel: float | None) -> str | None:
    """Why the reference shader's output `got` and the oracle's `want` disagree, or None."""
    assert got.shape == want.shape, label
    d = np.abs(got.astype(np.float64) - want)
    if rel is not None:
        r = d / (1.0 + np.abs(want))
        return None if r.max() < rel else f"{label}: max relative difference {r.max():.3e}"
    if label in TOLERATED:
        tol, frac = TOLERATED[label]
        return None if d.max() <= tol and (d > 0).mean() <= frac else f"{label}: max abs {d.max():.3e}, differing texels {(d > 0).mean():.3%}"
    if np.array_equal(np.ascontiguousarray(got).view(np.uint32), np.ascontiguousarray(want).view(np.uint32)):   # bit patterns: NaN == NaN
        return None
    return f"{label}: NOT bit-exact (max abs {d.max():.3e}, {(d > 0).mean():.3%} of values differ)"


def _check(case: str, res: dict, live: bool, rel: float | None = None) -> int:
    """`res`: {label: (reference shader output, oracle output)}; without the live shaders the first element is unused and the
    oracle is compared with the record of case `case`. Planes under TOLERATED, and every plane when `rel` is given, are compared
    with that tolerance; all others bit for bit."""
    bad = []
    if RECORDING:
        _recorded["planes"][case] = {label: _digest(got) for label, (got, _) in res.items()}
        for label, (got, _) in res.items():
            if rel is not None or label in TOLERATED:
                _recorded["samples"][f"{case}/{label}"] = _sample(got)
    record = _recorded if RECORDING else _load_record()
    digests = record["planes"].get(case, {})
    stale = [] if set(digests) == set(res) else [f"{case}: recorded planes {sorted(digests)} != compared planes {sorted(res)}"]
    for label, (got, want) in res.items():
        if live:
            why = _difference(label, got, want, rel)
            if label in digests and _digest(got) != digests[label]:
                stale.append(f"{case}/{label}: the reference shader's output differs from the record")
        elif label not in digests:
            continue
        elif rel is None and label not in TOLERATED:
            why = None if _digest(want) == digests[label] else f"{label}: NOT bit-exact (differs from the recorded output of the reference shader)"
        else:
            why = None if _digest(want) == digests[label] else _difference(label, record["samples"][f"{case}/{label}"], _sample(want), rel)
        if why:
            bad.append(why)
    assert not bad, "oracle differs from the reference's shaders:\n  " + "\n  ".join(bad)
    assert not stale, ("rewrite the record deliberately (DFX_RECORD_REFERENCE_SHADERS=1, see the module docstring):\n  " + "\n  ".join(stale))
    return len(res)


def test_default_chain_bit_exact(shaders):
    """The benchmarked configuration: every pass of PostFX, SSR, SSAO, TAA, Bloom and ToneMap, third frame of a sequence."""
    n = _check("default_chain", _run(Variant(), shaders), shaders)
    assert n >= 45


def test_reversed_depth_bit_exact(shaders):
    seq = [synth.reverse_depth_frame(f) for f in synth.generate_sequence(W, H, 3)]
    _check("reversed_depth", _run(Variant(reversed_depth=True), shaders, seq), shaders)


def test_half_resolution_bit_exact(shaders):
    _check("half_resolution", _run(Variant(ssr_flags=capi.SSR_FLAG_HALF_RESOLUTION, ssao_flags=capi.SSAO_FLAG_HALF_RESOLUTION), shaders), shaders)


def test_ssr_previous_frame_and_half_precision_depth_bit_exact(shaders):
    _check("ssr_previous_frame_ssao_half_precision", _run(Variant(ssr_flags=1, ssao_flags=1), shaders), shaders)


@pytest.mark.parametrize("algorithm", [1, 2], ids=["hbao", "vbao"])
def test_ssao_algorithms_bit_exact(shaders, algorithm):
    res = _run(Variant(ssao_algorithm=algorithm), shaders)
    _check(f"ssao_algorithm_{algorithm}", {k: v for k, v in res.items() if k.startswith("A")}, shaders)


@pytest.mark.parametrize("flags", [0, 1, 4, 5, 6, 7], ids=lambda f: f"taa_flags_{f}")
def test_taa_variants_bit_exact(shaders, flags):
    res = _run(Variant(taa_flags=flags), shaders)
    _check(f"taa_flags_{flags}", {k: v for k, v in res.items() if k.startswith("T")}, shaders)


@pytest.mark.parametrize("mode", [1, 2, 3, 5, 6, 7, 8, 9, 10, 11])
def test_tone_map_operators_bit_exact(shaders, mode):
    res = _run(Variant(tonemap_mode=mode, to_srgb=bool(mode & 1)), shaders, warm=0)
    _check(f"tone_map_{mode}", {k: v for k, v in res.items() if k.startswith("M")}, shaders)


def test_depth_of_field_bit_exact(shaders):
    a = capi.DOFAttribs.default()
    a.MaxCircleOfConfusion = 0.02
    frames = []
    for f in synth.generate_sequence(W, H, 3):
        g = dict(f)
        for k in ("curr_camera", "prev_camera"):
            c = capi.CameraAttribs.from_buffer_copy(bytes(f[k]))
            c.fFocusDistance, c.fFStop = 6.0, 1.4
            g[k] = c
        frames.append(g)
    for flags in (capi.DOF_FLAG_TEMPORAL_SMOOTHING | capi.DOF_FLAG_KARIS_INVERSE, 0):
        res = _run(Variant(dof=True, dof_flags=flags, dof_attribs=a), shaders, frames)
        assert any(k.startswith("D11") for k in res)
        _check(f"depth_of_field_flags_{flags}", {k: v for k, v in res.items() if k[0] in "DB"}, shaders)


@pytest.mark.parametrize("size", [(34, 18), (33, 17)], ids=["even", "odd"])
def test_bilateral_quad_derivatives_everywhere(shaders, size):
    """SSR_ComputeBilateralCleanup.fx takes ddx / ddy of the camera-space depth. With the filter branch live on EVERY pixel
    (the sequence tests reach it only where the variance is high) the oracle's 2x2 differences equal the shader's quad
    derivatives bit for bit - including, on odd-sized targets, the last column / row, whose quad partner lies outside the
    target: Direct3D runs it as a helper lane whose Load returns 0. (The oracle and dfx_ssr.cu used to clamp that partner onto
    the pixel itself; this comparison is what showed the difference, and both were changed to the Load-returns-0 rule.)"""
    from oracle import oracle_py as op
    w, h = size
    fr = synth.generate_sequence(w, h, 1)[0]
    rng = np.random.default_rng(1)
    ssr = capi.SSRAttribs.default()
    o = op.Oracle(w, h)
    o.set_ssr(ssr, 0)
    o.set_inputs(fr)
    depth = rng.uniform(0.3, 0.9, (h, w)).astype(np.float32)
    normal = np.zeros((h, w, 4), np.float32)
    normal[..., 2] = 1.0
    o.set("depth", depth), o.set("normal", normal), o.set("material", np.full((h, w, 4), 0.2, np.float32))
    o.run("ssr_mask")
    rough, mask = o.get("ssr_roughness"), o.get("ssr_mask")
    assert mask.all() and rough.min() >= 0.125                            # every pixel traced, full filter radius
    ci = fr["frame"] & 1
    rad, var = rng.uniform(0, 4, (h, w, 4)).astype(np.float32), np.ones((h, w), np.float32)
    o.set(f"ssr_radhist{ci}", rad), o.set(f"ssr_varhist{ci}", var)
    o.run("ssr_bilateral")
    want = o.get("ssr_out")
    assert np.abs(want - rad).max() > 0.1                                  # the filter really ran
    got = np.zeros_like(want)
    if shaders:
        refsh.run("ssr_bilateral", [depth, normal, rough, rad, var], [got], cbs=[fr["curr_camera"], ssr], mask=np.ones((h, w), np.uint8))
    _check(f"bilateral_{w}x{h}", {"S7 ssr_bilateral": (got, want)}, shaders)


@pytest.mark.parametrize("trial", range(6))
def test_random_configurations_bit_exact(shaders, trial):
    """Random frame size, scene seed, feature flags, tone-map operator and attribute values (seeded): every pass of the third frame
    must still equal its shader bit for bit."""
    rng = np.random.default_rng(2024 + trial)
    w, h = int(rng.integers(40, 220)), int(rng.integers(30, 130))
    v = Variant(ssr_flags=int(rng.integers(0, 4)), ssao_flags=int(rng.integers(0, 4)), ssao_algorithm=int(rng.integers(0, 3)), taa_flags=int(rng.integers(0, 8)),
                tonemap_mode=int(rng.integers(1, 12)), to_srgb=bool(rng.integers(0, 2)), dof=bool(rng.integers(0, 2)), dof_flags=int(rng.integers(0, 4)))
    if v.ssr_flags == 3:
        v.ssr_flags = 2                                   # the manifest builds previous-frame and half-resolution intersect separately
    if v.ssao_algorithm:
        v.ssao_flags = 0                                  # HBAO / VBAO are built for the full-resolution, full-precision path
    if v.ssao_flags == 3:
        v.ssao_flags = 2
    v.ssr.MostDetailedMip, v.ssr.MaxTraversalIntersections = int(rng.integers(0, 3)), int(rng.integers(8, 200))
    v.ssr.RoughnessThreshold, v.ssr.GGXImportanceSampleBias = float(rng.uniform(0.05, 0.6)), float(rng.uniform(0, 1))
    v.ssr.SpatialReconstructionRadius, v.ssao.SpatialReconstructionRadius = float(rng.uniform(0, 6)), float(rng.uniform(0, 6))
    v.ssao.EffectRadius, v.ssao.TemporalStabilityFactor = float(rng.uniform(0.2, 3)), float(rng.uniform(0, 1))
    v.bloom.Threshold, v.bloom.Intensity, v.bloom.Radius = float(rng.uniform(0, 2)), float(rng.uniform(0, 1)), float(rng.uniform(0.5, 1.0))
    v.taa.TemporalStabilityFactor, v.dof_attribs.MaxCircleOfConfusion = float(rng.uniform(0, 1)), float(rng.uniform(0.005, 0.03))
    seq = synth.generate_sequence(w, h, 3, seed=int(rng.integers(1, 1000)))
    if v.dof:
        focus, fstop = float(rng.uniform(2, 12)), float(rng.uniform(1.2, 8))
        lens = []
        for f in seq:
            g = dict(f)
            for k in ("curr_camera", "prev_camera"):
                c = capi.CameraAttribs.from_buffer_copy(bytes(f[k]))
                c.fFocusDistance, c.fFStop = focus, fstop
                g[k] = c
            lens.append(g)
        seq = lens
    assert _check(f"random_configuration_{trial}", _run(v, shaders, seq), shaders) >= 40


def test_brdf_table_bit_exact(shaders):
    """PrecomputeBRDF.psh against oracle_compose_ibl.cpp's brdf_lut(), at two sample counts."""
    from oracle import oracle_py as op
    o = op.Oracle(W, H)
    for size, samples, name in ((64, 512, "brdf_lut"), (32, 64, "brdf_lut__64")):     # powers of two, like the reference's 512 x 512 table
        o.brdf_lut(size, samples)
        want = o.get("brdf_lut")
        got = np.zeros_like(want)
        if shaders:
            refsh.run(name, [], [got])
        _check(f"brdf_table_{size}_{samples}", {f"BRDF table {size} x {size}, {samples} samples": (got, want)}, shaders)


@pytest.mark.parametrize("size", [(128, 64), (157, 89)], ids=["128x64", "157x89"])
def test_full_compose(shaders, size):
    """Hydrogent's HnPostProcess.psh (SSR re-weighted by the split-sum BRDF and exchanged for the specular IBL, then SSAO)
    against the oracle's compose_ibl, on planes that exercise opacity 0, out-of-range roughness and metals.

    The shader builds the view direction from the interpolated NDC position of the pixel; the runner interpolates it as
    -1 + 2 (x + 0.5) / W, the oracle as ((x + 0.5) / W - 0.5) / 0.5. For power-of-two sizes both are exact and the pass is
    bit-exact; for other sizes the last bit of the NDC position differs and the result agrees to 1e-5 (relative to 1 + |c|)."""
    from oracle import oracle_py as op
    w, h = size
    fr = synth.generate_sequence(w, h, 1)[0]
    rng = np.random.default_rng(5)
    color = fr["color"].copy()
    color[..., 3] = rng.choice([0.0, 0.35, 1.0], (h, w), p=[0.1, 0.2, 0.7])
    mat = fr["material"].copy()
    mat[..., 1] = rng.choice([0.0, 0.5, 1.0], (h, w))
    mat[..., 0] = np.where(rng.random((h, w)) < 0.05, 1.5, mat[..., 0])
    base = np.concatenate([rng.uniform(0.02, 1.0, (h, w, 3)), np.ones((h, w, 1))], -1).astype(np.float32)
    ibl = np.concatenate([np.exp2(rng.uniform(-4, 2, (h, w, 3))), np.ones((h, w, 1))], -1).astype(np.float32)
    ssr = np.concatenate([np.exp2(rng.uniform(-4, 3, (h, w, 3))), rng.uniform(0, 1, (h, w, 1))], -1).astype(np.float32)
    ao = rng.uniform(0.2, 1.0, (h, w)).astype(np.float32)
    o = op.Oracle(w, h)
    o.set_inputs(fr)
    o.brdf_lut(64, 512)
    lut = o.get("brdf_lut")
    for k, v in dict(color=color, material=mat, base_color=base, specular_ibl=ibl, ssr_out=ssr, ssao_out=ao).items():
        o.set(k, v)
    bits = lambda f: int(np.float32(f).view(np.uint32))  # noqa: E731
    res = {}
    for ssr_scale, ssao_scale in ((0.8, 0.6), (1.0, 0.0), (0.0, 1.0)):
        o.set_compose_scales(ssr_scale, ssao_scale)
        o.run("compose_ibl")
        want = o.get("composed")
        got = np.zeros_like(want)
        if shaders:
            refsh.run("compose_ibl", [color, ssr, ao, fr["normal"], ibl, mat, base, lut], [got], cbs=[fr["curr_camera"]], iparams=[bits(ssr_scale), bits(ssao_scale)])
        res[f"compose (SSRScale {ssr_scale}, SSAOScale {ssao_scale})"] = (got, want)
    pow2 = w & (w - 1) == 0 and h & (h - 1) == 0
    _check(f"compose_{w}x{h}", res, shaders, rel=None if pow2 else 1e-5)


# One pass that takes each structure as a constant buffer: (pass, inputs, outputs, the constant buffers it takes, slot of the structure).
def _cb_probes():
    d, d4 = np.full((8, 8), 0.5, np.float32), np.full((8, 8, 4), 0.5, np.float32)
    cam = synth.generate_sequence(8, 8, 1)[0]["curr_camera"]
    return {
        "CameraAttribs": ("postfx_reprojected_depth", [d], [d.copy()], [cam, cam], 0),
        "SSRAttribs": ("ssr_mask", [d4, d], [d.copy(), d.copy()], [capi.SSRAttribs.default()], 0),
        "SSAOAttribs": ("ssao_prefilter", [d], [d.copy()], [cam, capi.SSAOAttribs.default()], 1),
        "TAAAttribs": ("taa__b", [d4, d4, d4[..., :2].copy(), d, d], [d4.copy()], [cam, cam, capi.TAAAttribs.default()], 2),
        "BloomAttribs": ("bloom_prefilter", [d4], [d4.copy()], [capi.BloomAttribs.default()], 0),
        "ToneMapAttribs": ("tonemap__4", [d4], [d4.copy()], [capi.ToneMapAttribs.default()], 0),
        "DOFAttribs": ("dof_coc", [d], [d.copy()], [cam, capi.DOFAttribs.default()], 1),
    }


def _accepted_size(name, ins, outs, cbs, slot, iparams=()) -> int:
    """The size of the constant buffer in `slot` the reference's structure has: the harness refuses every other size (error 2)."""
    own = bytes(cbs[slot])
    for n in range(4, 2049, 4):
        probe = (C.c_uint8 * n).from_buffer_copy((own + bytes(n))[:n])
        try:
            refsh.run(name, ins, [o.copy() for o in outs], cbs=[probe if i == slot else c for i, c in enumerate(cbs)], iparams=iparams)
            return n
        except RuntimeError as e:
            assert "failed with 2" in str(e), e
    raise AssertionError(f"{name}: no constant-buffer size accepted in slot {slot}")


def test_constant_buffer_layouts_match_the_reference_structures(shaders):
    """Each harness memcpy's the C struct of include/dfx_b200.h into the structure the reference's .fxh declares and refuses
    (error 2) when the sizes differ; feeding a short struct must therefore fail, and the size it accepts for each structure is
    the size of the struct this project passes."""
    sizes = {}
    if shaders:
        class Short(C.Structure):
            _fields_ = [("x", C.c_float * 3)]

        d = np.zeros((8, 8), np.float32)
        with pytest.raises(RuntimeError, match="failed with 2"):
            refsh.run("postfx_reprojected_depth", [d], [d.copy()], cbs=[Short(), Short()])
        for struct, (name, ins, outs, cbs, slot) in _cb_probes().items():
            sizes[struct] = _accepted_size(name, ins, outs, cbs, slot, iparams=[0, 1] if name.startswith("tonemap") else ())
        if RECORDING:
            _recorded["constant_buffers"] = sizes
    recorded = (_recorded if RECORDING else _load_record())["constant_buffers"]
    assert not sizes or sizes == recorded, f"the reference's structures changed size: {sizes} (recorded: {recorded})"
    assert len(recorded) == 7 and {s: C.sizeof(getattr(capi, s)) for s in recorded} == recorded
