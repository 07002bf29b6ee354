"""Region reads from a compressed slide (``region.CompressedSlide``) at the bench size: a synthetic
tissue slide of 8192 chunks of 512^2 (64 chunks per row, net A) is compressed once, then

  (a) viewer windows: one 1024^2 window per call at seeded random positions;
  (b) patch batches: 256 random 256^2 patches per call (``read_regions``);
  (c) the same 1024^2 windows through the codec class, chunk by chunk (what zarr slicing does);
  (d) the whole slide through ``decompress_image`` into a page-locked array.

Every timed call ends in a device synchronise.  Windows of (a) are checked byte for byte against
the reconstruction of (d).  Prints one JSON line with the card name and power limit.

    python tools/regionbench.py [--chunks 8192] [--windows 50] [--batches 20] [--out r.json]
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import cae_oracle as O  # noqa: E402  (synthetic tiles + random-init checkpoint only)
from cnn_autoencoder_b200 import compress, decompress, _store  # noqa: E402
from cnn_autoencoder_b200._autoencoders import ConvolutionalAutoencoder  # noqa: E402
from cnn_autoencoder_b200.region import CompressedSlide  # noqa: E402


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        power = q[torch.cuda.current_device()] if q else 'unknown'
    except (OSError, subprocess.SubprocessError):
        power = 'unknown'
    return name, power


def timed(fn, n):
    times = []
    for _ in range(n):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    return times


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--chunks', type=int, default=8192)
    ap.add_argument('--gx', type=int, default=64, help='chunks per row')
    ap.add_argument('--ps', type=int, default=512)
    ap.add_argument('--arch', default='A')
    ap.add_argument('--batch-tiles', type=int, default=16)
    ap.add_argument('--windows', type=int, default=50)
    ap.add_argument('--batches', type=int, default=20)
    ap.add_argument('--codec-windows', type=int, default=3)
    ap.add_argument('--whole', type=int, default=2)
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
    base = tempfile.mkdtemp(prefix='regionbench_')
    try:
        path = os.path.join(base, 'slide.zarr')
        t0 = time.perf_counter()
        cs = compress.compress_image('CAE', chk, slide, path, patch_size=ps,
                                     batch_tiles=args.batch_tiles)
        t_compress = time.perf_counter() - t0
        del slide
        rng = np.random.default_rng(2026)
        win = 1024
        windows = [(int(rng.integers(0, H - win + 1)), int(rng.integers(0, W - win + 1)))
                   for _ in range(args.windows + 5)]
        patch_sets = [[(int(rng.integers(0, H - 256 + 1)), int(rng.integers(0, W - 256 + 1)))
                       for _ in range(256)] for _ in range(args.batches + 2)]
        out = dict(card=None, power_limit=None, arch=args.arch, chunks=gy * gx, ps=ps,
                   slide_px=[H, W], compress_s=round(t_compress, 3), bytes=cs['bytes'],
                   batch_tiles=args.batch_tiles)
        out['card'], out['power_limit'] = card()

        t0 = time.perf_counter()
        reader = CompressedSlide(path, chk, batch_tiles=args.batch_tiles)
        out['open_s'] = round(time.perf_counter() - t0, 3)

        # (a) viewer windows
        for y, x in windows[:5]:                                        # warm-up
            reader.read_region(y, x, win, win)
        it = iter(windows[5:])
        got_windows = []
        chunks_a = []

        def one_window():
            y, x = next(it)
            img = reader.read_region(y, x, win, win)
            if len(got_windows) < 4:
                got_windows.append(((y, x), img))
            chunks_a.append(reader.stats['decoded'])
        ta = timed(one_window, args.windows)
        out['a_viewer_1024'] = dict(calls=len(ta), windows_per_s=round(len(ta) / sum(ta), 2),
                                    MPps=round(len(ta) * win * win / 1e6 / sum(ta), 1),
                                    ms_median=round(1e3 * float(np.median(ta)), 2),
                                    ms_max=round(1e3 * max(ta), 2),
                                    chunks_per_call=round(float(np.mean(chunks_a)), 2),
                                    coder='device' if reader.stats['device_decoded'] else 'host')

        # (b) patch batches
        for boxes in patch_sets[:2]:
            reader.read_regions(boxes, 256, 256)
        itb = iter(patch_sets[2:])
        chunks_b, dev_b = [], []

        def one_batch():
            reader.read_regions(next(itb), 256, 256)
            chunks_b.append(reader.stats['decoded'])
            dev_b.append(reader.stats['device_decoded'])
        tb = timed(one_batch, args.batches)
        out['b_patches_256x256'] = dict(calls=len(tb), patches_per_call=256,
                                        patches_per_s=round(256 * len(tb) / sum(tb), 1),
                                        MPps=round(256 * len(tb) * 65536 / 1e6 / sum(tb), 1),
                                        ms_median=round(1e3 * float(np.median(tb)), 2),
                                        chunks_decoded_per_call=round(float(np.mean(chunks_b)), 1),
                                        device_coder_calls=int(sum(1 for d in dev_b if d)))

        # (c) the codec class, chunk by chunk (zarr's route), same windows as (a)
        codec = ConvolutionalAutoencoder(chk)
        arr = _store.DirArray(os.path.join(path, '0/0'), mode='r')

        def codec_window(y, x):
            img = np.empty((win, win, 3), dtype=np.uint8)
            for iy in range(y // ps, (y + win - 1) // ps + 1):
                for ix in range(x // ps, (x + win - 1) // ps + 1):
                    tile = codec.decode(arr.read_encoded((iy, ix, 0)))
                    a, b = max(y, iy * ps), min(y + win, (iy + 1) * ps)
                    c, d = max(x, ix * ps), min(x + win, (ix + 1) * ps)
                    img[a - y:b - y, c - x:d - x] = tile[a - iy * ps:b - iy * ps, c - ix * ps:d - ix * ps]
            return img
        codec_window(*windows[0])
        itc = iter(windows[5:])
        tc = timed(lambda: codec_window(*next(itc)), args.codec_windows)
        out['c_codec_class_1024'] = dict(calls=len(tc), windows_per_s=round(len(tc) / sum(tc), 3),
                                         MPps=round(len(tc) * win * win / 1e6 / sum(tc), 2),
                                         ms_median=round(1e3 * float(np.median(tc)), 1))

        # (d) the whole slide through decompress_image
        canvas = torch.empty((H, W, 3), dtype=torch.uint8).pin_memory().numpy()
        decompress.decompress_image(path, canvas, checkpoint=chk, batch_tiles=args.batch_tiles)
        td = timed(lambda: decompress.decompress_image(path, canvas, checkpoint=chk,
                                                       batch_tiles=args.batch_tiles), args.whole)
        out['d_decompress_image_whole'] = dict(calls=len(td), s_median=round(float(np.median(td)), 3),
                                               MPps=round(H * W / 1e6 / float(np.median(td)), 1))
        out['windows_equal_decompress_image'] = all(
            np.array_equal(img.cpu().numpy(), canvas[y:y + win, x:x + win]) for (y, x), img in got_windows)
        y, x = windows[5]
        out['codec_class_equal_decompress_image'] = bool(
            np.array_equal(codec_window(y, x), canvas[y:y + win, x:x + win]))
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
