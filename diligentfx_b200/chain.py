"""Python view of the chain-level C-ABI (`dfx_chain_*`): the full PostProcess chain of one view, one native call per frame.

The native executor mirrors the reference integration `HnPostProcessTask` (Hydrogent/src/Tasks/HnPostProcessTask.cpp): Prepare
(:591-683) prepares PostFXContext, SSR, SSAO, TAA, Bloom every frame; Execute (:743-947) runs
PostFX -> SSR -> SSAO -> compose -> TAA -> Bloom -> ToneMap(+sRGB). Sequencing, async-compute streams and CUDA-graph replay live
in libdfx_b200.so (csrc/dfx_effects.cu); this module owns the input / output device planes (torch tensors) and the host <->
device streaming pipeline of `stream_frames` (torch streams and events).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np
import torch

from . import capi
from .capi import BloomAttribs, Plane, Rows, SSAOAttribs, SSRAttribs, TAAAttribs, ToneMapAttribs, check, plane_of

STAGE_POSTFX, STAGE_SSR, STAGE_SSAO, STAGE_COMPOSE, STAGE_TAA, STAGE_BLOOM, STAGE_TONEMAP = 1, 2, 4, 8, 16, 32, 64
STAGE_ALL = 127

INPUT_SPECS = {  # name -> trailing channel count (0 = scalar plane)
    "depth": 0, "prev_depth": 0, "motion": 2, "normal": 4, "color": 4, "material": 4,
}
# Transfer formats of the G-buffer planes that are narrower than fp32 in the reference (Hydrogent/src/Tasks/HnBeginFrameTask.cpp:
# 63-68): input name -> (key in a packed frame, dtype, channels). Depth (D32_FLOAT) and the previous depth travel as fp32.
PACKED_SPECS = {
    "color": ("color16", torch.float16, 4), "normal": ("normal16", torch.float16, 4), "motion": ("motion16", torch.float16, 2),
    "material": ("material8", torch.uint8, 2),
}


def pack_frame(frame: dict, pin: bool = False) -> dict:
    """Host-side: a frame dict with the G-buffer in the reference's render-target formats (what a renderer would hand over).
    Colour is clamped to the half range; material keeps roughness (.x) and metallic (.y) as UNORM8."""
    out = {k: v for k, v in frame.items() if k not in PACKED_SPECS}
    for name, (key, dt, ch) in PACKED_SPECS.items():
        a = np.asarray(frame[name], np.float32)[..., :ch]
        if dt == torch.uint8:
            t = torch.from_numpy(np.floor(np.clip(a, 0.0, 1.0) * 255.0 + 0.5).astype(np.uint8))
        else:
            t = torch.from_numpy(np.clip(a, -65504.0, 65504.0).astype(np.float16))
        out[key] = t.contiguous().pin_memory() if pin else t.contiguous()
    for name in ("depth", "prev_depth"):
        t = frame[name] if isinstance(frame[name], torch.Tensor) else torch.from_numpy(np.ascontiguousarray(frame[name], np.float32))
        out[name] = t.pin_memory() if pin and not t.is_pinned() else t
    return out


def widen_frame(packed: dict) -> dict:
    """The fp32 frame dict the device sees after dfx_pass_unpack_plane (exact widening; material z = w = 0)."""
    out = {k: v for k, v in packed.items() if k not in {s[0] for s in PACKED_SPECS.values()}}
    for name, (key, dt, ch) in PACKED_SPECS.items():
        a = packed[key].numpy()
        if dt == torch.uint8:
            m = np.zeros(a.shape[:2] + (4,), np.float32)
            m[..., :ch] = a.astype(np.float32) / np.float32(255.0)
            out[name] = m
        else:
            out[name] = a.astype(np.float32)
    for name in ("depth", "prev_depth"):
        out[name] = packed[name].numpy() if isinstance(packed[name], torch.Tensor) else packed[name]
    return out


def pack_ldr8(ldr: np.ndarray) -> np.ndarray:
    """Host restatement of dfx_pass_pack_ldr8 (D3D UNORM rule: saturate, * 255, + 0.5, truncate; NaN -> 0)."""
    v = np.nan_to_num(np.asarray(ldr, np.float32), nan=0.0)
    # the kernel evaluates x * 255 + 0.5 as one fused multiply-add: exact in float64, rounded once to float32
    return (np.clip(v, 0.0, 1.0).astype(np.float64) * 255.0 + 0.5).astype(np.float32).astype(np.uint8)


@dataclass
class ChainConfig:
    ssao: SSAOAttribs = field(default_factory=SSAOAttribs.default)
    ssr: SSRAttribs = field(default_factory=SSRAttribs.default)
    bloom: BloomAttribs = field(default_factory=BloomAttribs.default)
    taa: TAAAttribs = field(default_factory=TAAAttribs.default)
    tonemap: ToneMapAttribs = field(default_factory=ToneMapAttribs.default)
    postfx_flags: int = 0                                  # capi.POSTFX_FLAG_REVERSED_DEPTH: the depth planes hold near = 1, far = 0
    ssao_flags: int = 0                                    # capi.SSAO_FLAG_HALF_RESOLUTION
    dof: capi.DOFAttribs | None = None                     # DepthOfField between TAA and Bloom (HnPostProcessTask.cpp:899-909); None = off
    dof_flags: int = 0                                     # capi.DOF_FLAG_TEMPORAL_SMOOTHING | capi.DOF_FLAG_KARIS_INVERSE
    ssr_flags: int = 0
    taa_flags: int = capi.TAA_FLAG_BICUBIC                 # Hydrogent default (HnPostProcessTask.hpp:109)
    ave_log_lum: float = 0.3                               # HnPostProcessTask.hpp:88, fExposure 0
    to_srgb: bool = True
    ssr_scale: float = 1.0
    ssao_scale: float = 1.0
    stages: int = STAGE_ALL
    fuse: bool = True          # compose inside TAA, ToneMap inside the Bloom composite (same per-pixel arithmetic, two HBM round trips fewer)
    overlap: bool = True       # async compute: SSAO beside SSR on a second stream, Bloom + ToneMap beside the NEXT frame's front half on a third
    graph: bool = True         # replay steady-state frames from CUDA graphs (dfx_chain_config.use_graph)
    # 0: tone-map with the constant ave_log_lum. capi.LUMINANCE_SAMPLING_REFERENCE (1) / _FULL (2): measure the scene's average luminance on
    # the device and tone-map with the adapted value when tonemap.bAutoExposure is set (tonemap.bLightAdaptation + the elapsed time adapt it)
    auto_exposure: int = 0


class PostProcessChain:
    """One view / one stream of consecutive frames on the current CUDA device: a thin view of the C-ABI's chain executor
    (`dfx_chain_*`, one call per frame). The executor sequences the effects like HnPostProcessTask, overlaps the SSAO passes
    with the SSR passes and Bloom + ToneMap with the next frame's front half on its own streams, and replays steady-state
    frames from CUDA graphs; this class only owns the input / output device planes (torch tensors)."""

    def __init__(self, width: int, height: int, config: ChainConfig | None = None, device: torch.device | None = None):
        self.lib = capi.load()
        self.w, self.h = width, height
        self.cfg = config or ChainConfig()
        self.device = device or torch.device("cuda", torch.cuda.current_device())
        if not torch.cuda.is_available():
            raise capi.DfxError("no CUDA device: the PostProcess chain has no CPU path")
        L = self.lib
        self._cfg_c = self._config_struct()
        self.chain = C.c_void_p()
        with torch.cuda.device(self.device):
            check(L.dfx_chain_create(width, height, C.byref(self._cfg_c), C.byref(self.chain)), "dfx_chain_create")
        fx = {n: C.c_void_p(L.dfx_chain_effect(self.chain, i)) for n, i in capi.CHAIN_EFFECT.items()}
        self.postfx, self.ssao, self.ssr, self.bloom, self.taa, self.dof = (fx[n] for n in ("postfx", "ssao", "ssr", "bloom", "taa", "dof"))
        dev = self.device
        # device-resident inputs (filled by upload()) and the LDR result
        self.inputs = {n: torch.empty((height, width) + ((c,) if c else ()), dtype=torch.float32, device=dev) for n, c in INPUT_SPECS.items()}
        self.ldr = torch.empty((height, width, 4), dtype=torch.float32, device=dev)
        self.frame_index = None
        self._post_stream = torch.cuda.ExternalStream(L.dfx_chain_post_stream(self.chain), device=dev)  # Bloom + ToneMap under cfg.overlap
        self._side_post = False

    def _config_struct(self) -> capi.ChainConfigC:
        cfg = self.cfg
        c = capi.ChainConfigC()
        c.ssao, c.ssr, c.bloom, c.taa, c.tonemap = cfg.ssao, cfg.ssr, cfg.bloom, cfg.taa, cfg.tonemap
        c.dof = cfg.dof if cfg.dof is not None else capi.DOFAttribs.default()
        c.postfx_flags, c.ssao_flags, c.ssr_flags, c.taa_flags, c.dof_flags = cfg.postfx_flags, cfg.ssao_flags, cfg.ssr_flags, cfg.taa_flags, cfg.dof_flags
        c.stages, c.enable_dof, c.fuse, c.overlap, c.use_graph, c.to_srgb = cfg.stages, int(cfg.dof is not None), int(cfg.fuse), int(cfg.overlap), int(cfg.graph), int(cfg.to_srgb)
        c.ave_log_lum, c.ssr_scale, c.ssao_scale = cfg.ave_log_lum, cfg.ssr_scale, cfg.ssao_scale
        c.auto_exposure = int(cfg.auto_exposure)
        return c

    def join(self):
        """Makes the current stream wait for everything execute(defer_post=True) left running on the executor's side stream."""
        check(self.lib.dfx_chain_join(self.chain, C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)), "dfx_chain_join")

    def stats(self) -> dict:
        s = capi.ChainStats()
        check(self.lib.dfx_chain_get_stats(self.chain, C.byref(s)))
        return {n: int(getattr(s, n)) for n, _ in s._fields_}

    def close(self):
        if getattr(self, "chain", None):
            self.lib.dfx_chain_destroy(self.chain)
        self.chain = self.postfx = self.ssao = self.ssr = self.bloom = self.taa = self.dof = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- input transfer -------------------------------------------------------------------------------------------
    def upload(self, frame: dict, non_blocking: bool = True) -> int:
        """Host (numpy or pinned torch) -> device copies of one frame's G-buffer. Returns bytes copied."""
        n = 0
        for name in INPUT_SPECS:
            src = frame[name]
            t = src if isinstance(src, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(src, np.float32))
            self.inputs[name].copy_(t, non_blocking=non_blocking)
            n += t.numel() * 4
        return n

    # ---- one frame ------------------------------------------------------------------------------------------------
    def set_elapsed_time(self, seconds: float):
        """Seconds since the previous frame (the reference's FrameAttribs.dElapsedTime) for light adaptation, from the next frame on."""
        check(self.lib.dfx_chain_set_elapsed_time(self.chain, float(seconds)), "dfx_chain_set_elapsed_time")

    def average_luminance(self) -> dict:
        """The auto-exposure state after the frames issued so far (synchronises the device): the adapted luminance as the R16F target
        holds it, the fAveLogLum the tone map used (max(0.05, state)), this frame's measurement exp(mean wlogL / mean w) and its weight."""
        torch.cuda.synchronize(self.device)
        out = download_plane(Plane(self.lib.dfx_chain_average_luminance_dev(self.chain), 16, 4, 1, capi.FORMAT_R32F, 0))[0]
        return {"state": float(out[0]), "ave_log_lum": float(out[1]), "measured": float(out[2]), "weight": float(out[3])}

    def execute(self, frame_index: int, curr_camera, prev_camera, inputs: dict | None = None, ldr_out: torch.Tensor | None = None,
                defer_post: bool = False, elapsed_time: float | None = None) -> torch.Tensor:
        """Runs the chain on device-resident inputs (default: the planes filled by upload()); returns the final LDR plane
        (device tensor, rgba; `ldr_out` if given). Everything is ordered after the work already on the current stream. With
        cfg.overlap the LDR plane is produced on a side stream: by default the current stream waits for it before this call
        returns; `defer_post=True` skips that wait so that the next frame's front half overlaps it (call join() before
        consuming the result). `elapsed_time`: seconds since the previous frame for light adaptation (kept for later frames;
        see set_elapsed_time)."""
        L, cfg = self.lib, self.cfg
        if elapsed_time is not None:
            self.set_elapsed_time(elapsed_time)
        c = self._config_struct()
        if bytes(c) != bytes(self._cfg_c):           # the caller edited self.cfg between frames
            self._cfg_c = c
            check(L.dfx_chain_set_config(self.chain, C.byref(c)), "dfx_chain_set_config")
        st = cfg.stages
        self._side_post = cfg.overlap and bool(st & STAGE_BLOOM) and bool(st & STAGE_TAA) and cfg.dof is None
        out = self.ldr if ldr_out is None else ldr_out
        P = {n: plane_of(t) for n, t in (inputs or self.inputs).items()}
        ldr = plane_of(out)
        fr = capi.ChainFrame(frame_index, int(defer_post), C.pointer(curr_camera), C.pointer(prev_camera), C.pointer(P["depth"]), C.pointer(P["prev_depth"]),
                             C.pointer(P["motion"]), C.pointer(P["normal"]), C.pointer(P["color"]), C.pointer(P["material"]), C.pointer(ldr))
        check(L.dfx_chain_execute(self.chain, C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream), C.byref(fr)), "dfx_chain_execute")
        self.frame_index = frame_index
        return out

    def run_frame(self, frame: dict) -> torch.Tensor:
        """Public one-call API: host G-buffer in, LDR device plane out (upload + execute)."""
        self.upload(frame)
        return self.execute(frame["frame"], frame["curr_camera"], frame["prev_camera"])

    def stream_frames(self, frames, ldr_host: list | None = None, packed: bool = False, new_sequence: bool = False,
                      elapsed_time: float | None = None) -> int:
        """Offline throughput path (BASELINE.json config 5: batches of frames): a double-buffered pipeline over three CUDA
        streams. While frame k runs on the compute stream, frame k+1's G-buffer is copied from (pinned) host memory on a
        copy stream and frame k-1's LDR result is copied back on a read-back stream; PCIe is full duplex, so the two copy
        directions overlap as well.

        `frames`: iterable of frame dicts (host planes + cameras + "frame" index). `ldr_host`: optional list of pinned
        (H, W, 4) float32 host tensors that receive the results (reused round-robin). Returns the number of frames run.

        `packed=True`: the frames carry the G-buffer in the reference's render-target formats (`pack_frame`: colour and
        normal RGBA16F, motion RG16F, material RG8; depths stay fp32) and `ldr_host` holds (H, W, 4) uint8 tensors: 30 B/px
        cross PCIe instead of 64, 4 B/px come back instead of 16. The passes read those formats directly (every half / UNORM8
        value is an fp32 value: the chain computes exactly what it computes on `widen_frame(packed_frame)`), so the narrow planes
        are also what the kernels pull from HBM.

        A frame without a "prev_depth" entry takes the depth of the frame streamed before it (its own depth if it is the
        first one), which stays on the device: in the reference the previous depth is last frame's depth target, not
        something the application uploads (HnPostProcessTask.cpp:788-832). Consecutive frames of one sequence then move 4 B/px less.
        The "frame streamed before" carries over from one call to the next unless `new_sequence=True`.

        `elapsed_time`: seconds between frames for light adaptation (cfg.auto_exposure); a frame's own "elapsed_time" entry wins.
        """
        dev = self.device
        if not hasattr(self, "_pipe"):
            mk = lambda: {n: torch.empty_like(t) for n, t in self.inputs.items()}  # noqa: E731
            self._pipe = dict(inputs=[mk(), mk()], ldr=[torch.empty_like(self.ldr), torch.empty_like(self.ldr)], h2d=torch.cuda.Stream(dev),
                              d2h=torch.cuda.Stream(dev), h2d_done=[torch.cuda.Event(), torch.cuda.Event()],
                              compute_done=[torch.cuda.Event(), torch.cuda.Event()], d2h_done=[torch.cuda.Event(), torch.cuda.Event()])
            self._pipe["depth_taken"] = [torch.cuda.Event(), torch.cuda.Event()]
            for e in self._pipe["compute_done"] + self._pipe["d2h_done"] + self._pipe["depth_taken"]:
                e.record(torch.cuda.current_stream(dev))
        P = self._pipe
        if packed and "staging" not in P:
            mk16 = lambda: {n: torch.empty((self.h, self.w, c), dtype=dt, device=dev) for n, (_, dt, c) in PACKED_SPECS.items()}  # noqa: E731
            P["staging"] = [mk16(), mk16()]
            P["ldr8"] = [torch.empty((self.h, self.w, 4), dtype=torch.uint8, device=dev) for _ in range(2)]
        main = torch.cuda.current_stream(dev)
        L, full = self.lib, Rows(0, self.h)
        if new_sequence:
            P["last_slot"] = None
        n = 0
        base = P.get("count", 0)                                     # slots keep alternating from one call to the next
        for k, fr in enumerate(frames):
            s = (base + k) & 1
            keep_prev = "prev_depth" not in fr                       # the previous depth stays on the device (see docstring)
            with torch.cuda.stream(P["h2d"]):
                P["h2d"].wait_event(P["compute_done"][s])          # frame k-2 no longer reads this input set
                P["h2d"].wait_event(P["depth_taken"][s])           # ... and frame k-1 has taken its previous depth from it
                for name in INPUT_SPECS:
                    if keep_prev and name == "prev_depth":
                        continue
                    if packed and name in PACKED_SPECS:
                        P["staging"][s][name].copy_(fr[PACKED_SPECS[name][0]], non_blocking=True)
                        continue
                    src = fr[name]
                    t = src if isinstance(src, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(src, np.float32))
                    P["inputs"][s][name].copy_(t, non_blocking=True)
                P["h2d_done"][s].record(P["h2d"])
            main.wait_event(P["h2d_done"][s])
            main.wait_event(P["d2h_done"][s])                        # frame k-2's result has left this LDR buffer
            if keep_prev:
                last = P.get("last_slot")
                P["inputs"][s]["prev_depth"].copy_(P["inputs"][s if last is None else last]["depth"])
                if last is not None:
                    P["depth_taken"][last].record(main)
            P["last_slot"] = s
            ins = P["inputs"][s]
            if packed:                                               # the passes read the render-target formats directly (Tex4 / Tex2 loaders): no widening pass
                ins = {n: (P["staging"][s][n] if n in PACKED_SPECS else t) for n, t in P["inputs"][s].items()}
            dt = fr.get("elapsed_time", elapsed_time)
            self.execute(fr["frame"], fr["curr_camera"], fr["prev_camera"], ins, ldr_out=P["ldr"][s], defer_post=True, elapsed_time=dt)
            # the frame is complete when its Bloom + ToneMap (side stream under cfg.overlap) is: the event goes on that stream
            post = self._post_stream if self._side_post else main
            if post is not main:
                post.wait_stream(main)
            result = P["ldr"][s]
            if packed:
                src, dst = plane_of(P["ldr"][s]), plane_of(P["ldr8"][s])
                check(L.dfx_pass_pack_ldr8(C.c_void_p(post.cuda_stream), C.byref(src), C.byref(dst), full), "dfx_pass_pack_ldr8")
                result = P["ldr8"][s]
            P["compute_done"][s].record(post)
            if ldr_host:
                with torch.cuda.stream(P["d2h"]):
                    P["d2h"].wait_event(P["compute_done"][s])
                    ldr_host[k % len(ldr_host)].copy_(result, non_blocking=True)
                    P["d2h_done"][s].record(P["d2h"])
            n += 1
        P["count"] = base + n
        self.join()
        main.wait_event(P["d2h_done"][0])
        main.wait_event(P["d2h_done"][1])
        return n

    # ---- debug access to effect-owned planes (parity tests) --------------------------------------------------------
    def fetch(self, effect: str, plane_id: int) -> np.ndarray:
        L = self.lib
        p = Plane()
        if effect == "postfx":
            check(L.dfx_postfx_get_plane(self.postfx, plane_id, C.byref(p)))
        elif effect == "ssao":
            check(L.dfx_ssao_get_plane(self.ssao, plane_id, C.byref(p)))
        elif effect == "ssr":
            check(L.dfx_ssr_get_plane(self.ssr, plane_id, C.byref(p)))
        elif effect == "bloom":
            check(L.dfx_bloom_get_plane(self.bloom, plane_id, C.byref(p)))
        elif effect == "taa":
            check(L.dfx_taa_get_plane(self.taa, plane_id, 0, C.byref(p)))
        elif effect == "dof":
            check(L.dfx_dof_get_plane(self.dof, plane_id, C.byref(p)))
        else:
            raise KeyError(effect)
        torch.cuda.synchronize(self.device)  # side streams included
        return download_plane(p)


def download_plane(p: Plane) -> np.ndarray:
    """Device plane -> numpy (H,W[,C]) float32 (uint8 masks are returned as float 0/1)."""
    L = capi.load()
    ch = {capi.FORMAT_R32F: 1, capi.FORMAT_RG32F: 2, capi.FORMAT_RGBA32F: 4, capi.FORMAT_R8U: 1}[p.format]
    if p.format == capi.FORMAT_R8U:
        out = np.empty((p.height, p.width), np.uint8)
    else:
        out = np.empty((p.height, p.width) if ch == 1 else (p.height, p.width, ch), np.float32)
    check(L.dfx_stream_synchronize(None))
    check(L.dfx_plane_download(None, C.byref(p), out.ctypes.data_as(C.c_void_p), 0), "dfx_plane_download")
    check(L.dfx_stream_synchronize(None))
    return out.astype(np.float32)
