#!/usr/bin/env python3
"""bench.py — Mpixels/s of the full PostProcess chain (PostFX prep -> SSR -> SSAO -> compose -> TAA -> Bloom -> ToneMap+sRGB)
on a synthetic 3840x2160 G-buffer (BASELINE.json metric / configs[2]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--width 3840 --height 2160] [--dump-outputs DIR]

One "step" = one frame of the chain. Rank r (one process per GPU; torchrun for N > 1) processes its own sequence of
frames: frames of a batch are independent sequences (SURVEY.md §8e, config 5: replicas, no data-path collective), so
scaling is weak and `value` = pixels all ranks processed / max-over-ranks device time.

Lines of the JSON record (one line on stdout, rank 0):
  value         device-resident throughput: the G-buffers of the timed steps are already in HBM in the renderer's formats (4 distinct
                frames, 0.22 GB each, cycled -> every step's inputs are cold in the 126 MB L2); timed with CUDA events, max over ranks.
                Async compute on three streams (ChainConfig.overlap; --no-overlap runs everything on one stream).
  e2e           the same K steps through the public streaming API (PostProcessChain.stream_frames) with HOST buffers: per
                step the frame's G-buffer is copied from pinned host memory in the reference's render-target formats
                (RGBA16F / RG16F / RG8 / D32F, which the passes read directly), the chain runs, and the frame is read back as RGBA8
                into pinned host memory; copy-in, compute and copy-out of neighbouring frames overlap on three streams.
                `e2e.fp32_transfers` is the same with every plane crossing PCIe as fp32.
  roofline      dominant pass of the chain (largest share of the step): algorithmic bytes / CUDA-event time inside this run
                (each pass alone on one stream), against MEASURED_PEAKS.json hbm_gbs (fallback 6650 GB/s,
                B200_PROFILING.md); `traffic` = DRAM bytes per launch from the committed ncu capture. `passes` lists every pass.
  cpu_baseline  the oracle (scalar C++ port of the Shaders/PostProcess math) on this box's host cores, bounded sample.
  --impl reference: the same metric from the reference's own pixel shaders compiled for the CPU (oracle/_ref, built from the HLSL
                sources by oracle/refshader; time inside the shader calls, all host cores), with the oracle port's number beside it
                in `port`; the port alone where oracle/_ref is absent. (The reference's C++ cannot be built here: DESIGN.md §2.)
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

def _baseline_metric() -> str:
    """The metric string of BASELINE.json, verbatim (falls back to its leading clause if the file is not around)."""
    try:
        return str(json.load(open(os.path.join(ROOT, "BASELINE.json")))["metric"])
    except Exception:
        return "Mpixels/sec full PostProcess chain @ 4K G-buffer"


METRIC = _baseline_metric()
UNIT = "Mpix/s"

# Algorithmic (compulsory) bytes per full-resolution pixel of each pass in this build's fp32 layout: every distinct plane the
# pass reads or writes counted once at its full size, pyramids as geometric sums (SURVEY.md §8d; derivation in DESIGN.md §4).
# G-buffer inputs in the renderer's formats (HnBeginFrameTask.cpp:63-69): colour / normal RGBA16F 8 B, motion RG16F 4 B, material RG8 2 B, depth 4 B.
PASS_BYTES_PER_PX = {
    "blue_noise": 0.0,
    "postfx_prepare": 28.0,              # depth 4 + previous depth 4 + motion 4 in; reprojected depth 4 + closest motion 8 + previous depth 4 out
    "ssr_hiz": 5.33, "ssr_mask_roughness": 11.0, "ssr_intersect": 58.33, "ssr_spatial": 73.0, "ssr_temporal": 77.0, "ssr_bilateral": 53.0,
    "ssao_prefilter_depth": 5.33, "ssao_ambient_occlusion": 17.33, "ssao_temporal": 36.0, "ssao_convolute": 10.67, "ssao_resample": 16.0,
    "ssao_spatial": 24.0,
    "compose": 44.0, "taa": 64.0,
    "compose_taa": 76.0,                 # fused: colour 8 + ssr 16 + ao 4 + history 16 + motion 8 + depths 8 in, accumulation 16 out
    "bloom_composite_tonemap": 36.0,     # fused: colour 16 + up[0] 4 in, LDR 16 out
    "bloom_prefilter": 20.0, "bloom_downsample": 6.67, "bloom_upsample": 12.0, "bloom_composite": 36.0, "bloom_tail": 0.0,   # pyramid entries: see bloom_bytes()
    "tonemap": 32.0,
    # DepthOfField (--dof only): CoC planes 4 B/px, half-size colour planes 16 B per quarter pixel
    "dof_coc": 8.0, "dof_temporal_coc": 20.0, "dof_separated_coc": 8.0, "dof_dilation": 6.6, "dof_blur_coc": 0.25, "dof_prefilter": 28.0,
    "dof_bokeh_first": 16.0, "dof_bokeh_second": 16.0, "dof_postfilter": 16.0, "dof_combine": 40.0,
}


# extra bytes per pixel when the G-buffer planes are widened to fp32 (--gbuffer fp32): colour / normal +8, motion +4, material +14
FP32_GBUFFER_EXTRA = {"postfx_prepare": 4.0, "ssr_mask_roughness": 14.0, "ssr_intersect": 16.0, "ssr_spatial": 8.0, "ssr_temporal": 4.0, "ssr_bilateral": 8.0,
                      "ssao_ambient_occlusion": 8.0, "ssao_spatial": 8.0, "compose": 8.0, "compose_taa": 8.0}


def bloom_bytes(W: int, H: int, mips: int, first: int) -> dict:
    """Exact algorithmic bytes of the Bloom pyramid passes from the level sizes (16 B texels): B2 per-level launches cover the levels
    1 .. first-1, the tail launch the levels first .. mips-1 down and mips-2 .. first-1 up, B3 per-level launches the levels first-2 .. 0."""
    lv = [(max((W // 2) >> i, 1), max((H // 2) >> i, 1)) for i in range(mips)]
    b = [16 * w * h for w, h in lv]
    top = mips - 1
    down = sum(b[i - 1] + b[i] for i in range(1, first))
    tail = b[first - 1] + sum(b[first:mips]) + sum(b[first - 1:top]) if first < mips else 0
    up = sum(2 * b[i - 1] + b[i] for i in range(min(top, first - 1), 0, -1))       # reads down[i-1] + coarser level, writes up[i-1]
    levels = sum(b[i - 1] + b[i] for i in range(1, mips)) + sum(2 * b[i - 1] + b[i] for i in range(top, 0, -1))   # dfx_pass_bloom_levels: all of B2 + B3
    return {"bloom_downsample": float(down), "bloom_tail": float(tail), "bloom_upsample": float(up), "bloom_levels": float(levels)}


def measured_hbm_peak() -> tuple[float, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(pass_name: str, width: int, height: int):
    """DRAM bytes per launch of the pass's kernel from the committed `ncu --set full` capture (profiles/r2d_ncu_traffic.json, made
    by tools/ncu_traffic_json.py from the raw page of the round-2 capture; G-buffer in the renderer formats),
    or None when the capture has no entry for it or was taken at another frame size (3840x2160)."""
    path = os.path.join(ROOT, "profiles", "r2d_ncu_traffic.json")
    try:
        d = json.load(open(path))
        k = d["kernels"][d["pass_to_kernel"][pass_name]]
    except (OSError, KeyError, ValueError):
        return None, "no ncu capture for this kernel"
    if (width, height) != (3840, 2160):
        return None, "ncu capture is for 3840x2160"
    return int(k["dram_bytes"]), "profiles/r2d_ncu_traffic.json (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch)"


def pin_to_gpu_numa_node(gpu_index: int) -> dict:
    """One process per GPU: run this rank's host threads on the CPU cores NVML reports as local to its GPU (same socket / NUMA node as
    the GPU's PCIe root), so that launches, pinned staging buffers and their first-touch pages do not cross the socket interconnect.
    Without it eight ranks share whatever cores the scheduler picks and the replicas lose ~12 % to host-side contention (round 1)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        n = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n)
        cpus = {64 * i + b for i, word in enumerate(mask) for b in range(64) if (word >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"cpus": len(cpus), "first": min(cpus), "last": max(cpus), "source": "nvmlDeviceGetCpuAffinity"}
    except Exception as e:  # no NVML / restricted container: keep the inherited affinity
        return {"cpus": len(os.sched_getaffinity(0)), "source": f"inherited ({type(e).__name__})"}
    return {"cpus": len(os.sched_getaffinity(0)), "source": "inherited"}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])), smax.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None, "reasons": sorted(reasons),
                "samples": len(sm)}


DUMP_PIXELS = 1 << 21   # 32 MB of RGBA float32


def dump_outputs(out_dir: str, ldr) -> None:
    """Writes what the timed path returned in its last step - the LDR plane of PostProcessChain.execute, RGBA float32 - as
    out_dir/ldr.npy with one row per pixel: the whole frame in raster order when it has at most DUMP_PIXELS pixels, else a fixed,
    seeded sample of DUMP_PIXELS of them (ascending raster index). The same --width / --height give the same pixels, so the
    files of two builds compare output for output."""
    import numpy as np
    import torch
    n = ldr.shape[0] * ldr.shape[1]
    idx = np.arange(n) if n <= DUMP_PIXELS else np.sort(np.random.default_rng(0).choice(n, DUMP_PIXELS, replace=False))
    rows = ldr.reshape(n, 4)[torch.from_numpy(idx).to(ldr.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "ldr.npy"), rows.astype(np.float32))


def cpu_baseline(width: int, height: int, frames: int, threads: int) -> dict:
    """Oracle full chain on a bounded sample (test infrastructure used as the reported CPU baseline only)."""
    from diligentfx_b200 import synth
    from oracle import oracle_py as op
    seq = synth.generate_sequence(width, height, frames)
    o = op.Oracle(width, height, threads=threads)
    times = []
    for fr in seq:
        o.set_inputs(fr)
        times.append(o.frame())
    steady = times[1:] if len(times) > 1 else times
    mpix = width * height / 1e6 / (statistics.median(steady) / 1e3)
    return {"value": round(mpix, 3), "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{len(steady)} consecutive {width}x{height} frames of the full chain (1/{(3840 * 2160) // (width * height)} of a 4K frame each), "
                      f"median; scalar C++ oracle (each pass bit-exact against the reference's own HLSL shader run on the CPU, "
                      f"tests/test_reference_shaders.py), rows dealt to a persistent std::thread pool"}


def psnr_vs_oracle(seq, W: int, H: int, threads: int) -> dict:
    """The metric's "PSNR vs ref" half: a FRESH chain and a fresh oracle both run the `len(seq)` consecutive frames of `seq`
    (frame 0 resets every history) at the benchmarked size; the last frame's planes are compared. LDR and AO: peak 1; HDR
    planes after Reinhard c/(1+c) (SURVEY.md 8d). Runs after the timed regions; the oracle here is the checker."""
    import numpy as np
    from diligentfx_b200.chain import PostProcessChain
    from oracle import oracle_py as op

    def psnr(a, b):
        mse = float(np.mean((np.asarray(a, np.float64) - np.asarray(b, np.float64)) ** 2))
        return 200.0 if mse == 0.0 else round(10.0 * np.log10(1.0 / mse), 2)

    def rh(x):
        x = np.maximum(np.nan_to_num(np.asarray(x, np.float64), nan=0.0, posinf=1e30), 0.0)
        return x / (1.0 + x)

    t0 = time.perf_counter()
    chain = PostProcessChain(W, H)          # the benchmarked configuration: fused passes, async compute
    o = op.Oracle(W, H, threads=threads)
    of = op.Oracle(W, H, threads=threads)   # the same chain with every render target rounded to the reference's texture format
    of.set_storage(True)
    for fr in seq:
        ldr = chain.run_frame(fr)
        for orc in (o, of):
            orc.set_inputs(fr)
            orc.frame()
    cur = seq[-1]["frame"] & 1
    got = ldr.cpu().numpy()
    want = o.get("ldr")
    out = {"ldr": psnr(np.clip(got[..., :3], 0, 1), np.clip(want[..., :3], 0, 1)),
           "ssao": psnr(chain.fetch("ssao", 0), o.get("ssao_out")),
           "ssr": psnr(rh(chain.fetch("ssr", 0)), rh(o.get("ssr_out"))),
           "taa": psnr(rh(chain.fetch("taa", 0)), rh(o.get(f"taa_accum{cur}"))),
           "bloom_up0": psnr(rh(chain.fetch("bloom", 30)[..., :3]), rh(o.get("bloom_up0")[..., :3])),
           "ldr_max_abs_err": float(np.abs(np.clip(got[..., :3], 0, 1) - np.clip(want[..., :3], 0, 1)).max()),
           # sensitivity (SURVEY.md Appendix B.5): how far the reference's own narrow render targets (R8 AO, RGBA16F SSR / TAA, R11G11B10F Bloom)
           # move the same frame - the kernels (fp32 planes) sit closer to the fp32 oracle than the reference's storage does
           "reference_storage_vs_fp32_ldr": psnr(np.clip(of.get("ldr")[..., :3], 0, 1), np.clip(want[..., :3], 0, 1)),
           "kernels_vs_reference_storage_ldr": psnr(np.clip(got[..., :3], 0, 1), np.clip(of.get("ldr")[..., :3], 0, 1)),
           "frames": len(seq), "size": [W, H], "floor_db": 49.0,
           "against": "the CPU oracle (each pass bit-exact against the reference's own HLSL shader, tests/test_reference_shaders.py), fp32 storage",
           "seconds": None}
    out["pass"] = bool(out["ldr"] >= 49.0)
    out["seconds"] = round(time.perf_counter() - t0, 1)
    chain.close()
    return out


def strips_leg(args, rank: int, world: int, dev) -> dict:
    """BASELINE.json config 4: ScreenSpaceReflection (S1-S7 + the PostFX planes it reads) on ONE 7680x4320 frame split into row strips
    over the ranks (strong scaling), through the native strips executor (halo rows pushed into the neighbours' slabs + flags, ray march
    and temporal history loaded from the owning GPU; no NCCL call per frame). Every rank also runs the unsharded frame sequence on its
    own GPU: its time is the 1-GPU reference of the speed-up, its output the bit-identity check of the rank's strip."""
    import numpy as np
    import torch
    import torch.distributed as dist

    from diligentfx_b200 import synth
    from diligentfx_b200.strips import SsrStrips, rebalance_bounds, reflective_block_cost, strip_bounds
    W8, H8, K, Wm = args.strips_width, args.strips_height, args.strips_steps, 3
    fr = synth.generate_sequence(W8, H8, 2, seed=11)[1]            # the same frame on every rank (second of a sequence: motion, previous camera)
    # cost-balanced strips: rays are only marched for reflective pixels, which a frame concentrates where its glossy surfaces are
    small = synth.generate_sequence(W8 // 8, H8 // 8, 2, seed=11)[1]
    refl = (small["material"][..., 0] <= 0.2) & (small["depth"] < 1.0 - 1e-6)
    bounds = strip_bounds(H8, world, weights=reflective_block_cost(refl.mean(axis=1), H8, march_cost=args.strips_march_cost)) if world > 1 else [(0, H8)]

    def run(x, frames: int, timed_from: int) -> float:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for i in range(frames):
            if i == timed_from:
                if world > 1:
                    dist.barrier()
                torch.cuda.synchronize()
                e0.record(x.stream)
            x.execute(i, fr["curr_camera"], fr["prev_camera"])
        e1.record(x.stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / (frames - timed_from)

    one = SsrStrips.virtual(W8, H8, [(0, H8)], dev)[0]              # unsharded: the same executor with one rank
    one.write_inputs(fr)
    ms1 = run(one, Wm + K, Wm)
    t = torch.tensor([ms1], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms1 = float(t.item())
    def profile(x, first: int) -> dict:
        """CUDA events around every pass and every exchange of 8 more frames (after the timed ones): ms per frame."""
        L = x.lib
        L.dfx_profile_reset()
        L.dfx_profile_enable(1)
        for i in range(8):
            x.execute(first + i, fr["curr_camera"], fr["prev_camera"])
        torch.cuda.synchronize()
        L.dfx_profile_enable(0)
        L.dfx_profile_collect()
        name, tot, calls = C.create_string_buffer(64), C.c_double(), C.c_int32()
        res = {}
        for i in range(L.dfx_profile_count()):
            L.dfx_profile_entry(i, name, 64, C.byref(tot), C.byref(calls))
            res[name.value.decode()] = round(tot.value / 8, 4)
        return res

    out = {"config": f"SSR S1-S7 + PostFX prep on one {W8}x{H8} frame (BASELINE.json configs[3]), inputs resident, {K} timed frames", "ms_1gpu": round(ms1, 4),
           "Mpix_s_1gpu": round(W8 * H8 / 1e6 / (ms1 / 1e3), 1)}
    if world > 1:
        # strips balanced by measurement: two rounds of (8 profiled frames -> per-rank compute time -> new cuts)
        sync_passes = ("strips_halo_wait", "strips_barrier_before_march", "strips_barrier_frame_end")
        slab, history = None, []
        for _ in range(args.strips_balance_rounds):
            x = SsrStrips.distributed(W8, H8, bounds, device=dev, slab=slab)
            x.write_inputs(fr)
            dist.barrier()
            for i in range(3):
                x.execute(i, fr["curr_camera"], fr["prev_camera"])
            p = profile(x, 3)
            mine_ms = [None] * world
            # what is balanced is the work AFTER the all-rank barrier (ray march .. bilateral cleanup): everything before it is levelled
            # by the barrier itself, so a rank with fewer rows gains nothing from finishing its part of it early
            # With many ranks the work BEFORE the barrier matters as well: it grows with a strip's rows (the top strip of this frame
            # is three times as tall as the others when only the post-barrier work is balanced, and everybody then waits for its PostFX /
            # Hi-Z / mask passes at the barrier: measured at N = 8), so from 4 ranks on the pre-march kernels count too.
            post = ("ssr_intersect_peer", "ssr_spatial", "ssr_temporal_peer", "ssr_bilateral", "strips_halo_push")
            pre = ("postfx_prepare", "ssr_hiz", "ssr_mask_roughness", "strips_gather_hiz") if world >= 4 else ()
            dist.all_gather_object(mine_ms, sum(v for k, v in p.items() if k in post + pre))
            history.append({"bounds": bounds, "compute_ms": [round(v, 3) for v in mine_ms]})
            bounds = rebalance_bounds(bounds, mine_ms, H8)
            slab = x.close(keep_slab=True)
        x = SsrStrips.distributed(W8, H8, bounds, device=dev, slab=slab)
        x.write_inputs(fr)
        dist.barrier()
        msn = run(x, Wm + K, Wm)
        t = torch.tensor([msn], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        msn = float(t.item())
        same = bool(np.array_equal(x.read("out"), one.read("out", rows=(x.y0, x.y1)))) and not x.timed_out()
        mine = profile(x, Wm + K)     # where the time goes, per rank (after the comparison: both executors have run the same frames until here)
        one_passes = profile(one, Wm + K)
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)
        ok = torch.tensor([1 if same else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        out.update({"n_gpus": world, "ms": round(msn, 4), "Mpix_s": round(W8 * H8 / 1e6 / (msn / 1e3), 1), "speedup": round(ms1 / msn, 3),
                    "efficiency": round(ms1 / msn / world, 3), "strips_bit_identical": bool(ok.item()), "bounds": bounds, "scaling": "strong",
                    "per_rank_pass_ms": per_rank, "one_gpu_pass_ms": one_passes, "balancing": history,
                    "exchange": "halo rows (64/4 depth, 4 normal + material, 1 motion; 4 ray planes; 1 resolved radiance; 2 radiance history) pushed into the neighbours' "
                                "slabs by a copy kernel + flags in peer memory; the Hi-Z pyramid all-gathered by peer stores before the march; colour / normal at ray hits and "
                                "last frame's history loaded from the owning GPU over NVLink; two all-rank flag barriers per frame; no NCCL call per frame"})
        x.close()
    one.close()
    return out


def _time_reference_shaders(seq, w: int, h: int, warmup: int, steps: int):
    """Seconds per frame spent inside the reference's own pixel shaders (oracle/_ref/librefshaders.so: the HLSL sources compiled
    for the CPU, every pass of the chain, all host cores), or None where that library is not available. The shaders are fed
    with the oracle's planes pass by pass (oracle/refshader/driver.py); only the shader calls are timed."""
    try:
        from oracle.refshader import refsh
        from oracle.refshader.driver import Variant, compare_frame, make_oracle
        if not refsh.available():
            return None
        v = Variant()
        o = make_oracle(w, h, v)
        acc = [0.0]
        real = refsh.run

        def timed(*a, **k):
            t0 = time.perf_counter()
            real(*a, **k)
            acc[0] += time.perf_counter() - t0

        refsh.run = timed
        try:
            for i in range(warmup + steps):
                fr = dict(seq[i % len(seq)])
                fr["frame"] = i
                if i < warmup:
                    o.set_inputs(fr)
                    o.frame()
                else:
                    compare_frame(o, fr, v)
        finally:
            refsh.run = real
        return acc[0] / steps
    except Exception as e:  # the arm must still print its line: fall back to the port
        sys.stderr.write(f"reference shaders not timed ({type(e).__name__}: {e}); using the oracle port\n")
        return None


def run_reference(args) -> None:
    """--impl reference. The reference has no CPU implementation of this path (its effects are GPU pixel shaders), but its shader
    sources compile for the CPU (oracle/refshader -> oracle/_ref): where that library is present the line's value is the
    throughput of those shaders on all host cores (`cpu_baseline.kind` "reference"), with the oracle port's throughput beside
    it in `port`; otherwise the port alone (`kind` "port")."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from diligentfx_b200 import synth
    from oracle import oracle_py as op
    threads = os.cpu_count() or 1
    w, h = args.ref_width, args.ref_height
    # like the GPU arm: a few distinct synthetic frames cycled under consecutive frame indices (histories stay live), so that
    # start-up does not grow with --steps
    seq = synth.generate_sequence(w, h, min(args.warmup + args.steps, args.frames))
    o = op.Oracle(w, h, threads=threads)
    t = 0.0
    for i in range(args.warmup + args.steps):
        fr = dict(seq[i % len(seq)])
        fr["frame"] = i
        o.set_inputs(fr)
        dt = o.frame()
        if i >= args.warmup:
            t += dt
    port_ms = t / args.steps
    port_value = w * h / 1e6 / (port_ms / 1e3)
    frame = f"each step = one {w}x{h} frame of the full chain (1/{(args.width * args.height) // (w * h)} of the {args.width}x{args.height} workload)"
    port = {"value": round(port_value, 3), "unit": UNIT, "ms_per_step": round(port_ms, 3), "cores": threads,
            "what": "the scalar C++ oracle port, each pass bit-exact against the reference's shaders (tests/test_reference_shaders.py), rows dealt to a persistent std::thread pool"}
    shader_s = _time_reference_shaders(seq, w, h, args.warmup, args.steps)
    if shader_s is not None:
        ms, kind = shader_s * 1e3, "reference"
        sample = (f"{frame}; the reference's own HLSL pixel shaders compiled for the CPU (oracle/_ref/librefshaders.so), every pass of the chain fed with the "
                  f"oracle's planes, time inside the shader calls only")
    else:
        ms, kind = port_ms, "port"
        sample = f"{frame}; the oracle port (the reference's shaders compiled for the CPU, oracle/_ref, are not available here)"
    value = w * h / 1e6 / (ms / 1e3)
    rec = {"impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"full PostProcess chain, {args.width}x{args.height} synthetic G-buffer (bounded sample: {sample})"},
           "cpu_baseline": {"value": round(value, 3), "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
           "port": port,
           "e2e": {"value": round(value, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(rec), flush=True)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--frames", type=int, default=4, help="distinct synthetic frames resident per rank (cycled)")
    ap.add_argument("--ref-width", type=int, default=960)
    ap.add_argument("--ref-height", type=int, default=540)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--psnr", action="store_true", help="run the PSNR-vs-oracle leg at N > 1 too (default: N = 1 only)")
    ap.add_argument("--no-psnr", action="store_true", help="skip the PSNR-vs-oracle leg (4 frames of the CPU oracle at the benchmarked size)")
    ap.add_argument("--no-overlap", action="store_true", help="run every pass on one stream (no async compute)")
    ap.add_argument("--no-strips", action="store_true", help="skip the row-strip leg (config 4: one 8K SSR frame split over the ranks)")
    ap.add_argument("--strips-only", action="store_true", help="only the row-strip leg (development: not the contract line)")
    ap.add_argument("--strips-n1", action="store_true", help="run the (unsharded) strips executor at N = 1 too")
    ap.add_argument("--strips-march-cost", type=float, default=13.0, help="cost of a reflective pixel relative to a plain one when the strips are balanced")
    ap.add_argument("--strips-balance-rounds", type=int, default=3, help="rounds of measured re-balancing of the strip boundaries before the timed run")
    ap.add_argument("--strips-width", type=int, default=7680)
    ap.add_argument("--strips-height", type=int, default=4320)
    ap.add_argument("--strips-steps", type=int, default=20)
    ap.add_argument("--gbuffer", default="native", choices=["native", "fp32"],
                    help="device-resident arm: G-buffer planes in the renderer's formats (RGBA16F / RG16F / RG8, what the passes read directly) or widened to fp32")
    ap.add_argument("--no-graph", action="store_true", help="issue every frame eagerly (no CUDA-graph replay)")
    ap.add_argument("--dof", action="store_true", help="add DepthOfField between TAA and Bloom (NOT the BASELINE.json workload; config.workload says so)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last one's LDR result to DIR/ldr.npy: RGBA float32, one row per pixel, "
                         "a fixed seeded sample of 2^21 pixels of larger frames")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)

    if args.impl == "reference":
        run_reference(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    from diligentfx_b200 import capi, synth
    from diligentfx_b200.chain import INPUT_SPECS, PACKED_SPECS, ChainConfig, PostProcessChain, pack_frame, widen_frame

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the chain has no CPU path (use --impl reference for the CPU oracle)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    all_cpus = os.sched_getaffinity(0)
    affinity = pin_to_gpu_numa_node(local_rank)   # before any pinned host buffer is allocated: first touch places it on this node
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"  # keep NCCL's version banner off stdout: rank 0 prints exactly one (JSON) line
        dist.init_process_group("nccl", device_id=dev)

    W, H, K, Wm = args.width, args.height, args.steps, args.warmup
    lib = capi.load()
    if args.strips_only:
        out = strips_leg(args, rank, world, dev)
        if rank == 0:
            print(json.dumps({"strips": out}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- synthetic data: `frames` consecutive frames of one camera path per rank ----
    # The renderer hands the G-buffer over in the reference's render-target formats (RGBA16F colour / normal, RG16F motion, RG8
    # material, D32F depths: Hydrogent/src/Tasks/HnBeginFrameTask.cpp:63-69); the fp32 planes the passes read are the exact
    # widening of those, on the device-resident arm as well, so both arms process the same values.
    seq = synth.generate_sequence(W, H, args.frames, seed=7)   # the same sequence on every rank: weak scaling means equal work per GPU (a seed per rank
    # made the ranks' frames differ in cost - reflective area - by several per cent, which the max-over-ranks time then read as a scaling loss)
    packed = [pack_frame(fr, pin=True) for fr in seq]
    seq = [widen_frame(p) for p in packed]
    host = [{n: torch.from_numpy(np.ascontiguousarray(fr[n])).pin_memory() for n in INPUT_SPECS} for fr in seq]
    # device-resident arm: the G-buffer lies in HBM in the renderer's formats (what `packed` holds) and the passes read it as such
    native = args.gbuffer == "native"
    resident = [{n: (packed[i][PACKED_SPECS[n][0]].to(dev) if (native and n in PACKED_SPECS) else host[i][n].to(dev)) for n in INPUT_SPECS} for i in range(len(host))]
    cams = [(fr["curr_camera"], fr["prev_camera"]) for fr in seq]
    # consecutive frames: the previous depth is the depth of the frame before and stays on the device (stream_frames docstring)
    packed = [{k: v for k, v in p.items() if k != "prev_depth"} for p in packed]
    packed_keys = [s[0] for s in PACKED_SPECS.values()] + ["depth"]
    h2d_bytes = sum(packed[0][k].numel() * packed[0][k].element_size() for k in packed_keys)
    h2d_bytes_fp32 = sum(t.numel() * 4 for t in host[0].values())
    dof = None
    if args.dof:  # not BASELINE.json's chain: Hydrogent's optional DepthOfField between TAA and Bloom, f/1.4 focused at 6 m
        dof = capi.DOFAttribs.default()
        dof.MaxCircleOfConfusion = 0.02
        for cp in cams:
            for c in cp:
                c.fFocusDistance, c.fFStop = 6.0, 1.4
    chain = PostProcessChain(W, H, ChainConfig(overlap=not args.no_overlap, graph=not args.no_graph, dof=dof, dof_flags=capi.DOF_FLAG_TEMPORAL_SMOOTHING if dof else 0), device=dev)
    ldr_host = torch.empty((H, W, 4), dtype=torch.float32).pin_memory()
    ldr8_hosts = [torch.empty((H, W, 4), dtype=torch.uint8).pin_memory() for _ in range(2)]
    d2h_bytes, d2h_bytes_fp32 = ldr8_hosts[0].numel(), ldr_host.numel() * 4

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    step_id = [0]

    def next_frame():
        # consecutive frame indices (histories stay valid); the resident G-buffers are cycled
        i = step_id[0]
        step_id[0] += 1
        return i, i % len(seq)

    def run_resident():
        idx, slot = next_frame()
        chain.execute(idx, cams[slot][0], cams[slot][1], resident[slot], defer_post=True)  # Bloom + ToneMap overlap the next frame's front half

    ldr_hosts = [ldr_host, torch.empty_like(ldr_host).pin_memory()]

    def e2e_frames(steps: int, src):
        # host frame dicts for the public streaming API: pinned G-buffer planes + cameras + consecutive frame index
        for _ in range(steps):
            idx, slot = next_frame()
            yield {**src[slot], "curr_camera": cams[slot][0], "prev_camera": cams[slot][1], "frame": idx}

    def run_e2e(steps: int):      # the G-buffer crosses PCIe in its render-target formats, the frame comes back as RGBA8
        chain.stream_frames(e2e_frames(steps, packed), ldr8_hosts, packed=True)

    def run_e2e_fp32(steps: int):  # everything crosses PCIe as fp32 (64 B/px in, 16 B/px out)
        chain.stream_frames(e2e_frames(steps, host), ldr_hosts)

    def timed(fn, steps: int, whole: bool = False) -> float:
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if whole:
            fn(steps)
        else:
            for _ in range(steps):
                fn()
        chain.join()                     # the side streams' work is inside the timed region
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- warm-up, then the timed device-resident region (clocks sampled during it) ----
    for _ in range(Wm):
        run_resident()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = lib.dfx_launch_count()
    total_ms = timed(run_resident, K)
    launches = lib.dfx_launch_count() - launches0
    issue = chain.stats()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, chain.ldr)   # before the legs below run more frames into the same plane
    ms_per_step = total_ms / K
    value = world * W * H / 1e6 / (ms_per_step / 1e3)

    # ---- end to end through the public API with host buffers ----
    run_e2e(3)
    e2e_ms = timed(run_e2e, K, whole=True) / K
    e2e_value = world * W * H / 1e6 / (e2e_ms / 1e3)
    run_e2e_fp32(3)
    e2e32_ms = timed(run_e2e_fp32, max(K // 4, 4), whole=True) / max(K // 4, 4)
    e2e32_value = world * W * H / 1e6 / (e2e32_ms / 1e3)

    # ---- per-pass device times (CUDA events on the launching stream, same steps) ----
    passes, roof = [], None
    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        lib.dfx_profile_reset()
        lib.dfx_profile_enable(1)
        overlap, chain.cfg.overlap = chain.cfg.overlap, False   # one stream: every pass is timed alone, back to back
        for _ in range(K):
            run_resident()
        torch.cuda.synchronize()
        chain.cfg.overlap = overlap
        lib.dfx_profile_enable(0)
        capi.check(lib.dfx_profile_collect())
        name, tot, calls = C.create_string_buffer(64), C.c_double(), C.c_int32()
        bloom_mips = lib.dfx_bloom_mip_count(W // 2, H // 2, C.c_float(chain.cfg.bloom.Radius))
        bloom_first = next((i for i in range(1, bloom_mips) if max((W // 2) >> i, 1) * max((H // 2) >> i, 1) <= 2048), bloom_mips)
        pyramid_bytes = bloom_bytes(W, H, bloom_mips, bloom_first if lib.dfx_tune_get(b"bloom_tail", 0) else bloom_mips)
        step_sum = 0.0
        for i in range(lib.dfx_profile_count()):
            capi.check(lib.dfx_profile_entry(i, name, 64, C.byref(tot), C.byref(calls)))
            nm = name.value.decode()
            ms = tot.value / K                                  # per step (a pass may launch several kernels / levels)
            step_sum += ms
            by = pyramid_bytes.get(nm, (PASS_BYTES_PER_PX.get(nm, 0.0) + (0.0 if native else FP32_GBUFFER_EXTRA.get(nm, 0.0))) * W * H)
            gbs = by / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
            passes.append({"pass": nm, "ms": round(ms, 4), "launch_groups_per_step": calls.value // K, "alg_bytes": int(by), "GBps": round(gbs, 1),
                           "frac": round(gbs / peak, 4)})
        for p in passes:
            p["share"] = round(p["ms"] / step_sum, 4) if step_sum else 0.0
        # The same, in the regime where the temporal filters are LIVE: the histories are reset every 4th frame (a jump of the frame
        # index), so the SSAO resampling / spatial reconstruction run their taps instead of the long-history early-out they take in
        # steady state (SSAO_ComputeSpatialReconstruction.fx:65-69, SSAO_ComputeResampledHistory.fx:67-71).
        lib.dfx_profile_reset()
        lib.dfx_profile_enable(1)
        chain.cfg.overlap = False
        base = step_id[0] + 1000
        for i in range(K):
            slot = i % len(seq)
            chain.execute(base + (i // 4) * 10 + (i % 4), cams[slot][0], cams[slot][1], resident[slot])
        torch.cuda.synchronize()
        chain.cfg.overlap = overlap
        lib.dfx_profile_enable(0)
        capi.check(lib.dfx_profile_collect())
        live = {}
        for i in range(lib.dfx_profile_count()):
            capi.check(lib.dfx_profile_entry(i, name, 64, C.byref(tot), C.byref(calls)))
            live[name.value.decode()] = tot.value / K
        step_id[0] = base + (K // 4 + 1) * 10
        for p in passes:
            if p["pass"] in live:
                ms = live[p["pass"]]
                p["live"] = {"ms": round(ms, 4), "frac": round(p["alg_bytes"] / (ms * 1e-3) / 1e9 / peak, 4) if ms > 0 else 0.0}
        top = max(passes, key=lambda p: p["ms"])
        traffic, traffic_src = ncu_traffic(top["pass"], W, H) if native else (None, "ncu capture is for the renderer-format G-buffer")
        roof = {"bound": "hbm", "kernel": top["pass"], "achieved": top["GBps"], "peak": peak, "unit": "GB/s", "frac": top["frac"], "traffic": traffic,
                "traffic_source": traffic_src, "alg_bytes": top["alg_bytes"], "peak_source": peak_src, "share_of_step": top["share"],
                "chain": {"alg_bytes_per_px": round(sum(p["alg_bytes"] for p in passes) / (W * H), 2),
                          "achieved": round(sum(p["alg_bytes"] for p in passes) / (ms_per_step * 1e-3) / 1e9, 1)}}
        roof["chain"]["frac"] = round(roof["chain"]["achieved"] / peak, 4)

    # ---- CPU baseline (rank 0, N = 1 only) ----
    os.sched_setaffinity(0, all_cpus)   # the CPU legs (oracle baseline, PSNR check) may use every host core again
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # a quarter of the workload's frame, 4 consecutive frames (median of the last 3): ~5-10 s on the GPU boxes' hosts. Larger than the
        # --impl reference arm's per-step sample on purpose: with 128 cores a 540-row frame leaves 4 rows per thread and times the pool.
        cpu = cpu_baseline(max(args.ref_width, 1920), max(args.ref_height, 1080), 4, os.cpu_count() or 1)
    quality = None
    if rank == 0 and not args.no_psnr and (world == 1 or args.psnr):   # one check per build: the N = 1 line carries it (N > 1 would idle N - 1 GPUs meanwhile)
        quality = psnr_vs_oracle([{**fr, "frame": i} for i, fr in enumerate(seq)], W, H, os.cpu_count() or 1)

    strips = None
    if not args.no_strips and (world > 1 or args.strips_n1):
        torch.cuda.empty_cache()
        strips = strips_leg(args, rank, world, dev)

    if rank == 0:
        rec = {
            "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": round(ms_per_step, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": ("NOT the BASELINE.json workload (--dof): DepthOfField added between TAA and Bloom; " if args.dof else "") +
                                   f"full PostProcess chain (PostFX prep, SSR, SSAO, compose, TAA bicubic, Bloom {lib.dfx_bloom_mip_count(W // 2, H // 2, C.c_float(0.75))} levels, "
                                   f"ToneMap Uncharted2 + sRGB) on a {W}x{H} synthetic G-buffer + history, consecutive frames, one sequence per GPU",
                       "width": W, "height": H, "parallelism": f"replicas x{world} (independent frame sequences, no data-path collective)",
                       "streams": ("3 per GPU: SSR chain + TAA | SSAO chain | Bloom + ToneMap (overlaps the next frame's front half); per-pass times in `passes` are "
                                   "measured serially on one stream, where the depth / AO pyramids use their single-launch TMA tile kernels; with the two halves "
                                   "side by side the executor issues them one launch per level (the frame is 1.7 % faster that way, profiles/r2k1b)"
                                   if chain.cfg.overlap else "1 per GPU"),
                       "issue": {**issue, "what": "frames replayed from CUDA graphs (steady state) vs issued eagerly, since the chain was created; "
                                                  "1 native call (dfx_chain_execute) per frame either way"},
                       "tune": os.environ.get("DFX_TUNE", ""), "host_affinity": affinity,
                       "gbuffer": ("renderer formats (colour / normal RGBA16F, motion RG16F, material RG8, depth R32F), read directly by the passes" if native
                                   else "widened to fp32 planes"),
                       "cache": f"{args.frames} distinct resident G-buffers of {h2d_bytes_fp32 / 1e6:.0f} MB cycled: inputs larger than the 126 MB L2"},
            "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": round(e2e_value, 2), "unit": UNIT, "ms_per_step": round(e2e_ms, 4), "h2d_bytes_per_step": int(h2d_bytes),
                    "d2h_bytes_per_step": int(d2h_bytes),
                    "h2d_GBps": round(h2d_bytes / (e2e_ms * 1e-3) / 1e9, 1),   # what bounds this number: the host link (PCIe 5 x16, ~55 GB/s achievable), not a kernel
                    "formats": "host G-buffer in the reference's render-target formats (RGBA16F colour / normal, RG16F motion, RG8 material, fp32 depth = "
                               "26 B/px; the previous depth is the depth of the frame before and stays on the device), read by the passes in those formats (no widening pass); result read back as RGBA8 (4 B/px); PostProcessChain.stream_frames("
                               "packed=True): copy-in / compute / copy-out pipelined on 3 streams",
                    "fp32_transfers": {"value": round(e2e32_value, 2), "ms_per_step": round(e2e32_ms, 4), "h2d_bytes_per_step": int(h2d_bytes_fp32),
                                       "d2h_bytes_per_step": int(d2h_bytes_fp32)}},
            "strips": strips, "psnr": quality, "roofline": roof, "cpu_baseline": cpu, "passes": passes,
        }
        print(json.dumps(rec), flush=True)
    chain.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
