#!/usr/bin/env python3
"""Run the chain over a few synthetic frames (a profiling target for ncu: few launches, no timing), or - with --in / --out - over a
directory of G-buffer frame files (diligentfx_b200/gbuffer_io.py: one .npz per frame in the renderer's formats), the offline-batch use of
BASELINE.json config 5: frames are streamed host -> device -> host through `PostProcessChain.stream_frames(packed=True)` in batches, the
RGBA8 results are written as .npy (or .ppm with --ppm).

    python tools/run_chain.py --write-synthetic /tmp/seq --width 1920 --height 1080 --frames 16     # make a sequence on disk (CPU only)
    python tools/run_chain.py --in /tmp/seq --out /tmp/seq_ldr                                      # B200
"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from diligentfx_b200 import gbuffer_io, synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--width", type=int, default=3840)
ap.add_argument("--height", type=int, default=2160)
ap.add_argument("--frames", type=int, default=3)
ap.add_argument("--write-synthetic", metavar="DIR", help="write the synthetic sequence as frame files and exit (no GPU needed)")
ap.add_argument("--in", dest="src", metavar="DIR", help="directory of .npz frames (one sequence, consecutive frame indices)")
ap.add_argument("--out", dest="dst", metavar="DIR", help="where the LDR frames go")
ap.add_argument("--batch", type=int, default=8, help="frames in flight per stream_frames call (pinned host buffers for that many results)")
ap.add_argument("--ppm", action="store_true", help="write binary PPM instead of .npy")
ap.add_argument("--auto-exposure", choices=("off", "reference", "full"), default="off",
                help="tone-map with the measured, adapted scene luminance: 64x64 samples as the reference takes them, or every pixel")
ap.add_argument("--frame-time", type=float, default=1.0 / 60.0, metavar="S", help="seconds between frames, for light adaptation (default 1/60)")
a = ap.parse_args()

if a.write_synthetic:
    os.makedirs(a.write_synthetic, exist_ok=True)
    for fr in synth.generate_sequence(a.width, a.height, a.frames):
        gbuffer_io.save_frame(os.path.join(a.write_synthetic, f"frame{fr['frame']:05d}.npz"), fr)
    print("wrote", a.frames, "frames to", a.write_synthetic)
    sys.exit(0)

from diligentfx_b200.chain import ChainConfig, PostProcessChain  # noqa: E402  (loads the CUDA library: fails loudly without it)

config = ChainConfig(auto_exposure={"off": 0, "reference": 1, "full": 2}[a.auto_exposure])

if a.src:
    if not a.dst:
        ap.error("--in needs --out")
    os.makedirs(a.dst, exist_ok=True)
    paths = gbuffer_io.sequence_paths(a.src)
    if not paths:
        ap.error(f"no .npz frames in {a.src}")
    first = gbuffer_io.load_frame(paths[0])
    h, w = first["depth"].shape
    chain = PostProcessChain(w, h, config)
    results = [torch.empty((h, w, 4), dtype=torch.uint8).pin_memory() for _ in range(a.batch)]
    done = 0
    for b0 in range(0, len(paths), a.batch):
        batch = [gbuffer_io.load_frame(p, pin=True) for p in paths[b0:b0 + a.batch]]
        n = chain.stream_frames(batch, ldr_host=results, packed=True, new_sequence=(b0 == 0), elapsed_time=a.frame_time)
        torch.cuda.synchronize()
        for k in range(n):
            name = os.path.splitext(os.path.basename(paths[b0 + k]))[0] + (".ppm" if a.ppm else ".npy")
            gbuffer_io.save_ldr(os.path.join(a.dst, name), results[k])
        done += n
    chain.close()
    print("done", done, "frames,", chain.lib.dfx_launch_count(), "launches")
else:
    seq = synth.generate_sequence(a.width, a.height, a.frames)
    chain = PostProcessChain(a.width, a.height, config)
    chain.set_elapsed_time(a.frame_time)
    for fr in seq:
        chain.run_frame(fr)
    torch.cuda.synchronize()
    print("done", chain.lib.dfx_launch_count(), "launches")
