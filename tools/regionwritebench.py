"""Region writes to a compressed slide (``region.CompressedSlide`` in mode 'r+', ``create_slide``)
at the bench size: a synthetic tissue slide of 8192 chunks of 512^2 (64 chunks per row, net A)
is compressed once, then

  (a) redaction: one 1024^2 window set to 0 per call at seeded random positions;
  (b) write-back: 256 non-overlapping random 256^2 patches per call (``write_regions`` from a
      CUDA tensor; the boxes are drawn by rejection sampling, since random boxes overlap);
  (c) the same redactions as (a) through the codec class, chunk by chunk (zarr's setitem:
      decode, paste, encode, write, one chunk at a time);
  (d) the whole slide built with ``create_slide`` from strips of 1, 4 and 16 chunk rows, against
      ``compress_image`` of the same slide; every chunk file checked byte for byte.

Every timed call ends in a device synchronise (and its files are written).  Prints one JSON
line with the card name and power limit.  Read numbers of the same slide: ``regionbench.py``.

    python tools/regionwritebench.py [--chunks 8192] [--redactions 30] [--batches 10] [--out r.json]
"""
import argparse
import hashlib
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

from oracle import cae_oracle as O  # noqa: E402  (synthetic tiles + random-init checkpoint only)
from cnn_autoencoder_b200 import compress, _store  # noqa: E402
from cnn_autoencoder_b200._autoencoders import ConvolutionalAutoencoder  # noqa: E402
from cnn_autoencoder_b200.region import CompressedSlide, create_slide  # noqa: E402
from tools.regionbench import card, timed  # noqa: E402


def digests(path):
    """name -> sha256 of every chunk file of the array at ``path``/0/0."""
    d = os.path.join(path, '0/0')
    return {f: hashlib.sha256(open(os.path.join(d, f), 'rb').read()).hexdigest()
            for f in os.listdir(d) if not f.startswith('.')}


def disjoint_boxes(rng, H, W, size, n):
    """``n`` random size x size boxes that share no pixel (rejection sampling)."""
    boxes = []
    while len(boxes) < n:
        y, x = int(rng.integers(0, H - size + 1)), int(rng.integers(0, W - size + 1))
        if all(abs(y - a) >= size or abs(x - b) >= size for a, b in boxes):
            boxes.append((y, x))
    return boxes


def stat_summary(times, px):
    return dict(calls=len(times), ms_median=round(1e3 * float(np.median(times)), 2),
                ms_max=round(1e3 * max(times), 2),
                MPps=round(len(times) * px / 1e6 / sum(times), 1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--chunks', type=int, default=8192)
    ap.add_argument('--gx', type=int, default=64, help='chunks per row')
    ap.add_argument('--ps', type=int, default=512)
    ap.add_argument('--arch', default='A')
    ap.add_argument('--batch-tiles', type=int, default=16)
    ap.add_argument('--redactions', type=int, default=30)
    ap.add_argument('--batches', type=int, default=10)
    ap.add_argument('--codec-windows', type=int, default=3)
    ap.add_argument('--strips', default='1,4,16', help='chunk rows per strip for (d)')
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
    base = tempfile.mkdtemp(prefix='regionwritebench_')
    out = dict(card=None, power_limit=None, arch=args.arch, chunks=gy * gx, ps=ps, slide_px=[H, W],
               batch_tiles=args.batch_tiles)
    out['card'], out['power_limit'] = card()
    try:
        path = os.path.join(base, 'slide.zarr')
        compress.compress_image('CAE', chk, slide, path, patch_size=ps, batch_tiles=args.batch_tiles)
        rng = np.random.default_rng(2026)
        win = 1024
        windows = [(int(rng.integers(0, H - win + 1)), int(rng.integers(0, W - win + 1)))
                   for _ in range(args.redactions + args.codec_windows + 3)]
        patch_sets = [disjoint_boxes(rng, H, W, 256, 256) for _ in range(args.batches + 1)]

        t0 = time.perf_counter()
        slide_w = CompressedSlide(path, chk, batch_tiles=args.batch_tiles, mode='r+')
        out['open_s'] = round(time.perf_counter() - t0, 3)

        # (a) redactions
        slide_w[windows[0][0]:windows[0][0] + win, windows[0][1]:windows[0][1] + win] = 0  # warm-up
        it = iter(windows[3:3 + args.redactions])
        st_a = []

        def one_redaction():
            y, x = next(it)
            slide_w[y:y + win, x:x + win] = 0
            st_a.append(dict(slide_w.stats))
        ta = timed(one_redaction, args.redactions)
        out['a_redact_1024'] = dict(stat_summary(ta, win * win),
                                    chunks_per_call=round(float(np.mean([s['chunks'] for s in st_a])), 2),
                                    full_per_call=round(float(np.mean([s['full'] for s in st_a])), 2),
                                    coder='device' if st_a[-1]['device_coded'] else 'host')

        # (b) write-back of patch batches
        vals = torch.randint(0, 256, (256, 256, 256, 3), dtype=torch.uint8, device='cuda')
        slide_w.write_regions(patch_sets[0], 256, 256, vals)                           # warm-up
        itb = iter(patch_sets[1:])
        st_b = []

        def one_batch():
            slide_w.write_regions(next(itb), 256, 256, vals)
            st_b.append(dict(slide_w.stats))
        tb = timed(one_batch, args.batches)
        out['b_patches_256x256'] = dict(stat_summary(tb, 256 * 256 * 256), patches_per_call=256,
                                        patches_per_s=round(256 * len(tb) / sum(tb), 1),
                                        chunks_per_call=round(float(np.mean([s['chunks'] for s in st_b])), 1),
                                        device_coded_calls=int(sum(1 for s in st_b if s['device_coded'])))
        slide_w.close()

        # (c) the codec class, chunk by chunk (zarr's setitem), the windows after those of (a)
        codec = ConvolutionalAutoencoder(chk)
        arr = _store.DirArray(os.path.join(path, '0/0'), mode='r')

        def codec_redaction(y, x):
            for iy in range(y // ps, (y + win - 1) // ps + 1):
                for ix in range(x // ps, (x + win - 1) // ps + 1):
                    a, b = max(y, iy * ps), min(y + win, (iy + 1) * ps)
                    c, d = max(x, ix * ps), min(x + win, (ix + 1) * ps)
                    if b - a == ps and d - c == ps:
                        tile = np.zeros((ps, ps, 3), dtype=np.uint8)
                    else:
                        tile = codec.decode(arr.read_encoded((iy, ix, 0))).copy()
                        tile[a - iy * ps:b - iy * ps, c - ix * ps:d - ix * ps] = 0
                    arr.write_encoded((iy, ix, 0), codec.encode(tile))
        codec_redaction(*windows[1])
        itc = iter(windows[3 + args.redactions:])
        tc = timed(lambda: codec_redaction(*next(itc)), args.codec_windows)
        out['c_codec_class_redact_1024'] = stat_summary(tc, win * win)

        # (d) the whole slide from strips against compress_image
        ref_path = os.path.join(base, 'ref.zarr')
        t0 = time.perf_counter()
        compress.compress_image('CAE', chk, slide, ref_path, patch_size=ps, batch_tiles=args.batch_tiles)
        torch.cuda.synchronize()
        out['d_compress_image_s'] = round(time.perf_counter() - t0, 3)
        ref = digests(ref_path)
        ref_meta = open(os.path.join(ref_path, '0/0/.zarray')).read()
        shutil.rmtree(ref_path)
        built = os.path.join(base, 'built.zarr')
        for rows in (int(r) for r in args.strips.split(',')):
            s = create_slide(built, chk, slide.shape, patch_size=ps, overwrite=True,
                             batch_tiles=args.batch_tiles)
            step = rows * ps
            per_call = []
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for y0 in range(0, H, step):
                t1 = time.perf_counter()
                s[y0:y0 + step] = slide[y0:y0 + step]
                per_call.append(time.perf_counter() - t1)
            torch.cuda.synchronize()
            total = time.perf_counter() - t0
            coder = 'device' if s.stats['device_coded'] else 'host'
            s.close()
            same = digests(built) == ref and open(os.path.join(built, '0/0/.zarray')).read() == ref_meta
            out['d_strips_%d_rows' % rows] = dict(
                calls=len(per_call), chunks_per_call=rows * gx, s_total=round(total, 3),
                ms_per_call_median=round(1e3 * float(np.median(per_call)), 2),
                MPps=round(H * W / 1e6 / total, 1), coder=coder, files_equal_compress_image=same)
            shutil.rmtree(built)
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
