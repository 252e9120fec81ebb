"""Row-strip sharded SSR (native executor `dfx_ssr_strips_*`: halo rows pushed into the neighbours' slabs and announced by flags, ray
march and temporal history loaded from the owning rank) must be BIT-IDENTICAL to the unsharded run of the same kernels (SURVEY.md 8e).

* `test_virtual_ranks_*`: all ranks in one process on ONE GPU, one stream each - the same kernels, flags and peer addressing as the
  multi-GPU run, so the driver's single-GPU test pass covers the sharding logic (strip bookkeeping, halo widths, odd-height Hi-Z levels,
  ping-pong histories, flag protocol).
* `test_two_gpus_*`: one process per GPU over CUDA IPC + NVLink (needs >= 2 devices: `gpurun --gpus 2`).

Rows a rank does not own are poisoned (NaN inputs) until an exchange fills them: a missing or too narrow exchange shows up as NaN /
a differing texel in the owned rows. Frame height 432 = 6.75 blocks of 64 rows: Hi-Z levels 216, 108, 54, 27, 13, 6 - two odd-height
levels whose last row of a strip reads one row of the next block (the case round 1 got wrong).
"""
import os
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W, H, FRAMES = 320, 432, 3


def _reference(seq):
    from diligentfx_b200.chain import STAGE_POSTFX, STAGE_SSR, ChainConfig, PostProcessChain
    ref = PostProcessChain(W, H, ChainConfig(stages=STAGE_POSTFX | STAGE_SSR))
    for fr in seq:
        ref.run_frame(fr)
    out = {"out": ref.fetch("ssr", 0), "radiance": ref.fetch("ssr", 3), "resolved_radiance": ref.fetch("ssr", 5)}
    ref.close()
    return out


def _poisoned(fr, y0, y1):
    """The frame with every row this rank does not own replaced by NaN."""
    out = dict(fr)
    for n in ("depth", "prev_depth", "motion", "normal", "color", "material"):
        a = np.full_like(np.asarray(fr[n], np.float32), np.nan)
        a[y0:y1] = fr[n][y0:y1]
        out[n] = a
    return out


@pytest.mark.parametrize("bounds", [[(0, 192), (192, 432)], [(0, 128), (128, 320), (320, 432)], [(0, 64), (64, 64), (64, 432)]],
                         ids=["2 ranks", "3 ranks", "3 ranks, one empty"])
def test_virtual_ranks_bit_identical(built, bounds):
    import torch

    from diligentfx_b200 import synth
    from diligentfx_b200.strips import SsrStrips
    seq = synth.generate_sequence(W, H, FRAMES)
    want = _reference(seq)
    ranks = SsrStrips.virtual(W, H, bounds)
    try:
        for fr in seq:
            for x in ranks:
                x.write_inputs(_poisoned(fr, x.y0, x.y1), rows=(0, H))  # the whole plane: own rows valid, everything else NaN
            torch.cuda.synchronize()
            for x in ranks:
                x.execute(fr["frame"], fr["curr_camera"], fr["prev_camera"])
            torch.cuda.synchronize()
        assert not any(x.timed_out() for x in ranks), "a flag wait timed out: an exchange was never signalled"
        for name in ("radiance", "resolved_radiance", "out"):
            for x in ranks:
                if x.y1 == x.y0:
                    continue
                got = x.read(name)
                assert np.isfinite(got).all(), f"{name}: poison leaked into rank {x.rank}'s rows"
                assert np.array_equal(got, want[name][x.y0:x.y1]), f"{name}: rank {x.rank} differs from the unsharded frame (max abs {np.abs(got - want[name][x.y0:x.y1]).max()})"
    finally:
        for x in ranks:
            x.close()


def _free_port() -> int:
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank: int, world: int, port: int, out_dir: str):
    import torch
    import torch.distributed as dist

    from diligentfx_b200 import synth
    from diligentfx_b200.strips import SsrStrips, strip_bounds
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        seq = synth.generate_sequence(W, H, FRAMES)
        bounds = strip_bounds(H, world, weights=[1.0, 3.0, 3.0, 3.0, 3.0, 3.0, 3.0])  # unequal, cost-balanced strips
        x = SsrStrips.distributed(W, H, bounds)
        for fr in seq:
            x.write_inputs(_poisoned(fr, x.y0, x.y1), rows=(0, H))
            dist.barrier()  # the test poisons the halo rows from the host: nobody may have pushed into them yet
            x.execute(fr["frame"], fr["curr_camera"], fr["prev_camera"])
            torch.cuda.synchronize()
            dist.barrier()
        assert not x.timed_out()
        np.save(os.path.join(out_dir, f"strip_{rank}.npy"), x.read("out"))
        if rank == 0:
            np.save(os.path.join(out_dir, "ref.npy"), _reference(seq)["out"])
        x.close()
    finally:
        dist.destroy_process_group()


def test_two_gpus_bit_identical(built, tmp_path):
    import torch
    import torch.multiprocessing as mp

    from diligentfx_b200.strips import strip_bounds
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    if not torch.cuda.can_device_access_peer(0, 1):
        pytest.skip("GPUs 0 and 1 have no peer path")
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    ref = np.load(tmp_path / "ref.npy")
    for r, (y0, y1) in enumerate(strip_bounds(H, world, weights=[1.0, 3.0, 3.0, 3.0, 3.0, 3.0, 3.0])):
        got = np.load(tmp_path / f"strip_{r}.npy")
        assert np.isfinite(got).all(), "poison rows leaked into the owned strip: an exchange is missing"
        assert np.array_equal(got, ref[y0:y1]), f"strip {r} differs from the single-GPU result (max abs {np.abs(got - ref[y0:y1]).max()})"
