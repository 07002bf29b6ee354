"""Reduced-resolution region reads (``CompressedSlide.downsampled``) at the bench size: the slide,
net and conventions of ``regionbench.py`` (8192 chunks of 512^2, 64 chunks per row, net A,
random-init seed 1234, ``batch_tiles`` 16), then

  (a) viewer windows: one 1024^2 window of the level image per call, at f = 4 and 16;
  (b) patch batches: 256 random 256^2 patches of the level image per call, at f = 2 and 4;
  (c) the outputs of (a) and (b) through the route without this feature: ``read_region(s)`` at
      level 0, then an exact int32 reshape-sum-round in torch on the device (the windows are
      block-aligned, so the bytes must equal (a) and (b));
  (d) a whole-slide thumbnail at f = 64 (``downsampled(64)[:]``, a host ndarray), against
      ``decompress_image`` into a page-locked array followed by PIL's ``Image.reduce`` on the host;
  (e) the kernel alone: CUDA-event time of ``cae_tiles_crop_reduce_u8`` on one batch of 16
      decoded 512^2 tiles (L2-resident, as after the synthesis) for every f, and of the level-0
      crop kernel on the same batch.

Every timed call ends in a device synchronise.  Peak device memory per call is
``torch.cuda.max_memory_allocated`` above what was allocated before the call.  Prints one JSON
line with the card name and power limit.

    python tools/regionreducebench.py [--chunks 8192] [--windows 20] [--batches 10] [--out r.json]
"""
import argparse
import ctypes
import json
import os
import shutil
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
from PIL import Image  # noqa: E402

from oracle import cae_oracle as O  # noqa: E402  (synthetic tiles + random-init checkpoint only)
from cnn_autoencoder_b200 import _cabi as C, compress, decompress  # noqa: E402
from cnn_autoencoder_b200.region import CompressedSlide  # noqa: E402
from tools.regionbench import card  # noqa: E402


def torch_reduce(t, f):
    """Block means of ``t`` (... x H x W x c uint8 on the device, H and W multiples of f), rounded
    half up: the reduction torch offers for uint8 is a sum with an int32 accumulator."""
    *lead, H, W, c = t.shape
    s = t.view(*lead, H // f, f, W // f, f, c).sum(dim=(-4, -2), dtype=torch.int32)
    return ((s + f * f // 2) // (f * f)).to(torch.uint8)


def measure(fn, items):
    """Per call: seconds (ending in a device synchronise) and peak device bytes above the start."""
    times, peaks = [], []
    for item in items:
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        t0 = time.perf_counter()
        out = fn(item)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
        peaks.append(torch.cuda.max_memory_allocated() - base)
        del out
    return times, peaks


def summary(times, peaks, **extra):
    return dict(calls=len(times), ms_median=round(1e3 * float(np.median(times)), 2),
                ms_max=round(1e3 * max(times), 2),
                peak_MB=round(max(peaks) / 2 ** 20, 1), **extra)


def kernel_times(reader, tiles, f, reps):
    """CUDA-event time per launch of the reduce kernel (crop kernel for f = 0) on ``tiles``."""
    n, ps, _, c = tiles.shape
    lc = ps // max(f, 1)
    if f:
        pieces = np.array([[k, k, 0, 0, 0, 0, lc, lc, ps, ps, 0, 0] for k in range(n)], dtype=np.int32)
    else:
        pieces = np.array([[k, k, 0, 0, 0, 0, ps, ps] for k in range(n)], dtype=np.int32)
    out = torch.empty((n, lc, lc, c), dtype=torch.uint8, device='cuda')
    pdev = torch.empty(pieces.size, dtype=torch.int32, device='cuda')
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def launch():
        if f:
            C.check(C.lib().cae_tiles_crop_reduce_u8(tiles.data_ptr(), n, ps, c, f, pieces.ctypes.data,
                                                     n, pdev.data_ptr(), out.data_ptr(), n, lc, lc, st))
        else:
            C.check(C.lib().cae_tiles_crop_u8(tiles.data_ptr(), n, ps, c, pieces.ctypes.data, n,
                                              pdev.data_ptr(), out.data_ptr(), n, lc, lc, st))
    for _ in range(20):
        launch()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        launch()
    b.record()
    torch.cuda.synchronize()
    if f:   # the last launch's output against torch on the same tiles
        assert torch.equal(out, torch_reduce(tiles, f))
    return 1e3 * a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--chunks', type=int, default=8192)
    ap.add_argument('--gx', type=int, default=64, help='chunks per row')
    ap.add_argument('--ps', type=int, default=512)
    ap.add_argument('--arch', default='A')
    ap.add_argument('--batch-tiles', type=int, default=16)
    ap.add_argument('--windows', type=int, default=20)
    ap.add_argument('--batches', type=int, default=10)
    ap.add_argument('--whole', type=int, default=2)
    ap.add_argument('--kernel-reps', type=int, default=200)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    ps, gx = args.ps, args.gx
    gy = -(-args.chunks // gx)
    H, W = gy * ps, gx * ps
    bank = {(i, j): O.synth_tissue_tile(i, j, ps=ps, seed=3) for i in range(4) for j in range(4)}
    slide = np.empty((H, W, 3), dtype=np.uint8)
    for i in range(gy):
        for j in range(gx):
            slide[i * ps:(i + 1) * ps, j * ps:(j + 1) * ps] = bank[(i % 4, j % 4)]
    chk = O.make_checkpoint(O.NAMED_ARCHS[args.arch], seed=1234)
    base = tempfile.mkdtemp(prefix='regionreducebench_')
    try:
        path = os.path.join(base, 'slide.zarr')
        cs = compress.compress_image('CAE', chk, slide, path, patch_size=ps,
                                     batch_tiles=args.batch_tiles)
        del slide
        out = dict(card=None, power_limit=None, arch=args.arch, chunks=gy * gx, ps=ps,
                   slide_px=[H, W], bytes=cs['bytes'], batch_tiles=args.batch_tiles)
        out['card'], out['power_limit'] = card()
        reader = CompressedSlide(path, chk, batch_tiles=args.batch_tiles)
        rng = np.random.default_rng(2026)
        same = {}

        # (a) viewer windows and (c) the same windows through a level-0 read
        win = 1024
        for f in (4, 16):
            view = reader.downsampled(f)
            ly, lx = view.shape[:2]
            wins = [(int(rng.integers(0, ly - win + 1)), int(rng.integers(0, lx - win + 1)))
                    for _ in range(args.windows + 2)]
            for y, x in wins[:2]:                                             # warm-up
                view.read_region(y, x, win, win)
            got, chunks = [], []

            def one(yx):
                img = view.read_region(yx[0], yx[1], win, win)
                chunks.append(reader.stats['decoded'])
                if len(got) < 3:
                    got.append((yx, img.cpu()))
                return img
            t, p = measure(one, wins[2:])
            out['a_viewer_1024_f%d' % f] = summary(
                t, p, MPps_level=round(len(t) * win * win / 1e6 / sum(t), 1),
                MPps_level0=round(len(t) * (win * f) ** 2 / 1e6 / sum(t), 1),
                chunks_per_call=round(float(np.mean(chunks)), 1),
                coder='device' if reader.stats['device_decoded'] else 'host')
            n_c = min(len(wins) - 2, max(3, args.windows // 4))
            t, p = measure(lambda yx: torch_reduce(
                reader.read_region(yx[0] * f, yx[1] * f, win * f, win * f), f), wins[2:2 + n_c])
            out['c_level0_then_torch_1024_f%d' % f] = summary(t, p)
            same['a_f%d' % f] = all(torch.equal(torch_reduce(reader.read_region(
                y * f, x * f, win * f, win * f), f).cpu(), img) for (y, x), img in got)

        # (b) patch batches and (c) the same patches through level-0 patches
        pw = 256
        for f in (2, 4):
            view = reader.downsampled(f)
            ly, lx = view.shape[:2]
            sets = [[(int(rng.integers(0, ly - pw + 1)), int(rng.integers(0, lx - pw + 1)))
                     for _ in range(256)] for _ in range(args.batches + 2)]
            for boxes in sets[:2]:
                view.read_regions(boxes, pw, pw)
            chunks = []

            def batch(boxes):
                r = view.read_regions(boxes, pw, pw)
                chunks.append(reader.stats['decoded'])
                return r
            t, p = measure(batch, sets[2:])
            out['b_patches_256_f%d' % f] = summary(
                t, p, patches_per_s=round(256 * len(t) / sum(t), 1),
                chunks_per_call=round(float(np.mean(chunks)), 1),
                coder='device' if reader.stats['device_decoded'] else 'host')
            lvl0 = lambda boxes: [(y * f, x * f) for y, x in boxes]  # noqa: E731
            t, p = measure(lambda boxes: torch_reduce(
                reader.read_regions(lvl0(boxes), pw * f, pw * f), f), sets[2:])
            out['c_level0_then_torch_256_f%d' % f] = summary(t, p)
            same['b_f%d' % f] = bool(torch.equal(view.read_regions(sets[2], pw, pw), torch_reduce(
                reader.read_regions(lvl0(sets[2]), pw * f, pw * f), f)))

        # (d) whole-slide thumbnail at f = 64
        f = 64
        thumb = reader.downsampled(f)[:]
        t, p = measure(lambda _: reader.downsampled(f)[:], range(args.whole))
        out['d_thumbnail_f64'] = summary(t, p, s_median=round(float(np.median(t)), 3),
                                         chunks=reader.stats['decoded'],
                                         device_decoded=reader.stats['device_decoded'])
        canvas = torch.empty((H, W, 3), dtype=torch.uint8).pin_memory().numpy()

        pil_s, small = [], []

        def via_decompress(_):
            decompress.decompress_image(path, canvas, checkpoint=chk, batch_tiles=args.batch_tiles)
            t1 = time.perf_counter()
            small[:] = [np.asarray(Image.fromarray(canvas).reduce(f))]
            pil_s.append(time.perf_counter() - t1)
        via_decompress(None)
        t, _ = measure(via_decompress, range(args.whole))
        out['d_decompress_image_then_pil_f64'] = dict(
            calls=len(t), s_median=round(float(np.median(t)), 3),
            pil_reduce_s_median=round(float(np.median(pil_s[1:])), 3))
        # 65536 x 32768 is a multiple of 64: every block is full, where PIL is exact
        same['d_f64_pil'] = bool(np.array_equal(thumb, small[0]))
        del canvas

        # (e) the kernel alone on one batch of 16 decoded tiles
        n = args.batch_tiles
        side = int(np.sqrt(n))
        blk = reader.read_region(0, 0, side * ps, (n // side) * ps)
        tiles = blk.view(side, ps, n // side, ps, 3).permute(0, 2, 1, 3, 4).contiguous().view(n, ps, ps, 3)
        fs = [1 << i for i in range(int(np.log2(ps)) + 1)]
        out['e_kernel_us_per_batch'] = {'crop_f1': round(kernel_times(reader, tiles, 0, args.kernel_reps), 2)}
        for f in fs:
            out['e_kernel_us_per_batch']['reduce_f%d' % f] = round(
                kernel_times(reader, tiles, f, args.kernel_reps), 2)
        out['e_batch_MB'] = round(tiles.numel() / 1e6, 2)
        out['outputs_equal'] = same
        reader.close()
    finally:
        shutil.rmtree(base, ignore_errors=True)
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
