#!/usr/bin/env python3
"""Cost of auto exposure on a B200, in one call: the luminance passes alone (CUDA events) and the device-resident 4K chain frame with
dfx_chain_config.auto_exposure 0 / 1 / 2, alternated round by round in the same process. Writes a JSON under profiles/ (or --out) with
the card's name and power limit read in the same call.

    python tools/bench_auto_exposure.py [--width 3840 --height 2160 --iters 200 --rounds 5 --frames 20] [--out profiles/x.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from diligentfx_b200 import capi, synth  # noqa: E402
from diligentfx_b200.chain import ChainConfig, PostProcessChain  # noqa: E402

HBM_PEAK = 7.7e12  # bytes/s, NVIDIA HGX B200 data sheet, one GPU


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[torch.cuda.current_device()]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def time_pass(fn, iters):
    for _ in range(10):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / iters * 1e3  # us


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--frames", type=int, default=20, help="timed chain frames per configuration and round")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "auto_exposure_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_auto_exposure needs a CUDA device: there is nothing to measure on the CPU")
    w, h = a.width, a.height
    L = capi.load()
    res = {"card": card(), "width": w, "height": h}

    # ---- the passes alone (colour plane larger than L2 at 4K RGBA32F: 133 MB; RGBA16F: 66 MB)
    rng = np.random.default_rng(1)
    col32 = torch.from_numpy(np.exp2(rng.uniform(-6, 4, (h, w, 4))).astype(np.float32)).cuda()
    col16 = col32.half()
    state = torch.zeros(capi.AVERAGE_LUMINANCE_STATE_FLOATS, dtype=torch.float32, device="cuda")
    sp = C.c_void_p(state.data_ptr())
    capi.check(L.dfx_pass_reset_average_luminance(None, sp))
    tm = capi.ToneMapAttribs.default()
    passes = {}
    for name, t, sampling in (("full_rgba32f", col32, 2), ("full_rgba16f", col16, 2), ("reference_rgba32f", col32, 1)):
        p = capi.plane_of(t)
        fn = lambda p=p, s=sampling: capi.check(L.dfx_pass_update_average_luminance(None, C.byref(tm), s, C.c_float(1 / 60), C.byref(p), sp))  # noqa: E731
        us = time_pass(fn, a.iters)
        entry = {"us": round(us, 2)}
        if sampling == 2:
            nbytes = w * h * t.element_size() * 4
            entry.update(bytes=nbytes, achieved_TBps=round(nbytes / (us * 1e-6) / 1e12, 3), share_of_hbm_peak=round(nbytes / (us * 1e-6) / HBM_PEAK, 3))
        passes[name] = entry
    res["passes"] = passes

    # ---- the device-resident chain frame, auto_exposure 0 / 1 / 2 alternated
    seq = synth.generate_sequence(w, h, 2)
    chains = {ae: PostProcessChain(w, h, ChainConfig(auto_exposure=ae)) for ae in (0, 1, 2)}
    for ch in chains.values():
        ch.upload(seq[0])
        ch.set_elapsed_time(1 / 60)
    fidx = {ae: 0 for ae in chains}
    times = {ae: [] for ae in chains}

    def run(ae, n):
        ch, fr = chains[ae], seq[0]
        for _ in range(n):
            ch.execute(fidx[ae], fr["curr_camera"], fr["prev_camera"], defer_post=True)
            fidx[ae] += 1
        ch.join()

    for ae in chains:
        run(ae, 10)  # warm-up: graphs built
    torch.cuda.synchronize()
    for _ in range(a.rounds):
        for ae in chains:
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            run(ae, a.frames)
            t1.record()
            torch.cuda.synchronize()
            times[ae].append(t0.elapsed_time(t1) / a.frames)
    res["chain_frame_ms"] = {f"auto_exposure_{ae}": {"median": round(float(np.median(v)), 4), "min": round(min(v), 4), "max": round(max(v), 4),
                                                     "rounds": [round(x, 4) for x in v], "stats": chains[ae].stats()} for ae, v in times.items()}
    base = float(np.median(times[0]))
    res["chain_overhead_ms"] = {f"auto_exposure_{ae}": round(float(np.median(times[ae])) - base, 4) for ae in (1, 2)}
    res["note"] = ("pass times: CUDA events over back-to-back launches; chain: 4K device-resident frames, async compute + graphs, frame rate "
                   "of a steady stream of frames (defer_post), median of the rounds; the spread of auto_exposure_0 bounds the noise")
    for ch in chains.values():
        ch.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
