"""Resolution pyramids (``CompressedSlide.build_pyramid``, ``level(k)``) at the bench size: the
slide, net and conventions of ``regionbench.py`` (8192 chunks of 512^2, 64 chunks per row, net A,
random-init seed 1234, ``batch_tiles`` 16), then

  (a) ``build_pyramid()`` at the default K (7 here): wall time and peak device memory, beside the
      peak of a whole-slide ``downsampled(64)[:]`` read;
  (b) the route without this feature: for every k, ``downsampled(2^k)[:]`` and ``compress_image``
      of that level image; the level files of (a) and (b) must be byte-identical, every level;
  (c) viewer windows of 1024^2 at 1/4 and 1/16 through ``level(2)`` and ``level(4)``, against
      ``downsampled(4)`` and ``downsampled(16)`` (the chunk counts are asserted);
  (d) the kernel alone: CUDA-event time of ``cae_tiles_pyramid_u8`` on one L2-resident batch of
      16 decoded 512^2 tiles, all 7 levels, over ``--kernel-reps`` launches.

Every timed call ends in a device synchronise.  Peak device memory per call is
``torch.cuda.max_memory_allocated`` above what was allocated before the call.  Prints one JSON
line with the card name and power limit.

    python tools/pyramidbench.py [--chunks 8192] [--windows 20] [--out r.json]
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

from oracle import cae_oracle as O  # noqa: E402  (synthetic tiles + random-init checkpoint only)
from cnn_autoencoder_b200 import _cabi as C, compress  # noqa: E402
from cnn_autoencoder_b200.region import CompressedSlide  # noqa: E402
from tools.regionbench import card  # noqa: E402
from tools.regionreducebench import measure, summary  # noqa: E402


def level_files(path, k):
    d = os.path.join(path, '0', str(k))
    return {f: open(os.path.join(d, f), 'rb').read() for f in sorted(os.listdir(d))}


def kernel_time(tiles, levels, reps):
    """CUDA-event time per launch of the pyramid kernel on ``tiles`` (n x ps x ps x c, one row)."""
    n, ps, _, c = tiles.shape
    recs = np.array([[0, j, ps, ps] for j in range(n)], dtype=np.int32)
    width = sum(-(-n // 2 ** k) for k in range(1, levels + 1))
    out = torch.zeros((width, ps, ps, c), dtype=torch.uint8, device='cuda')
    rdev = torch.empty(recs.size, dtype=torch.int32, device='cuda')
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def launch():
        C.check(C.lib().cae_tiles_pyramid_u8(tiles.data_ptr(), n, ps, c, levels, recs.ctypes.data,
                                             rdev.data_ptr(), 1, n, out.data_ptr(), st))
    for _ in range(20):
        launch()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        launch()
    b.record()
    torch.cuda.synchronize()
    return 1e3 * a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--chunks', type=int, default=8192)
    ap.add_argument('--gx', type=int, default=64, help='chunks per row')
    ap.add_argument('--ps', type=int, default=512)
    ap.add_argument('--arch', default='A')
    ap.add_argument('--batch-tiles', type=int, default=16)
    ap.add_argument('--windows', type=int, default=20)
    ap.add_argument('--builds', type=int, default=3)
    ap.add_argument('--kernel-reps', type=int, default=500)
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
    base = tempfile.mkdtemp(prefix='pyramidbench_')
    try:
        path = os.path.join(base, 'slide.zarr')
        cs = compress.compress_image('CAE', chk, slide, path, patch_size=ps,
                                     batch_tiles=args.batch_tiles)
        del slide
        out = dict(card=None, power_limit=None, arch=args.arch, chunks=gy * gx, ps=ps,
                   slide_px=[H, W], bytes=cs['bytes'], batch_tiles=args.batch_tiles)
        out['card'], out['power_limit'] = card()
        reader = CompressedSlide(path, chk, batch_tiles=args.batch_tiles, mode='r+')
        same = {}

        # (a) the build, repeated with overwrite=True (the first call is the warm-up)
        reader.build_pyramid(overwrite=True)
        K = max(reader.levels)
        t, p = measure(lambda _: reader.build_pyramid(overwrite=True), range(args.builds))
        out['a_build_pyramid'] = summary(t, p, s_median=round(float(np.median(t)), 3), levels=K,
                                         decoded=reader.stats['decoded'],
                                         level_chunks=reader.stats['level_chunks'],
                                         device_coded=reader.stats['device_coded'])
        built = {k: level_files(path, k) for k in range(1, K + 1)}
        t, p = measure(lambda _: reader.downsampled(64)[:], range(2))
        out['a_thumbnail_downsampled64'] = summary(t, p, decoded=reader.stats['decoded'])

        # (b) every level through downsampled(2^k)[:] and compress_image
        ref = os.path.join(base, 'ref')
        per_level = {}

        def route_b(_):
            for k in range(1, K + 1):
                t0 = time.perf_counter()
                img = reader.downsampled(2 ** k)[:]
                compress.compress_image('CAE', chk, img, os.path.join(ref, str(k)), patch_size=ps,
                                        batch_tiles=args.batch_tiles)
                per_level[k] = round(time.perf_counter() - t0, 3)
        t, p = measure(route_b, range(1))
        out['b_downsampled_then_compress_image'] = dict(s=round(t[0], 3), peak_MB=round(p[0] / 2 ** 20, 1),
                                                        s_per_level=per_level)
        for k in range(1, K + 1):
            d = os.path.join(ref, str(k), '0', '0')
            same['level%d_files' % k] = built[k] == {
                f: open(os.path.join(d, f), 'rb').read() for f in sorted(os.listdir(d))}

        # (c) viewer windows at 1/4 and 1/16: the stored level against the reduced read
        rng = np.random.default_rng(2026)
        win = 1024
        for k in (2, 4):
            f = 2 ** k
            ly, lx = reader.level(k).shape[:2]
            wins = [(int(rng.integers(0, ly - win + 1)), int(rng.integers(0, lx - win + 1)))
                    for _ in range(args.windows + 2)]
            for name, view in (('stored_level%d' % k, reader.level(k)),
                               ('downsampled%d' % f, reader.downsampled(f))):
                for y, x in wins[:2]:
                    view.read_region(y, x, win, win)
                chunks = []

                def one(yx):
                    img = view.read_region(yx[0], yx[1], win, win)
                    chunks.append(reader.stats['decoded'])
                    return img
                t, p = measure(one, wins[2:])
                out['c_viewer_1024_f%d_%s' % (f, name)] = summary(
                    t, p, chunks_per_call=round(float(np.mean(chunks)), 1), chunks_max=max(chunks))
                if name.startswith('stored'):
                    assert max(chunks) <= 9, chunks          # a 1024^2 window spans <= 3 x 3 chunks

        # (d) the kernel alone on one batch of 16 decoded tiles (L2-resident)
        n = args.batch_tiles
        side = int(np.sqrt(n))
        blk = reader.read_region(0, 0, side * ps, (n // side) * ps)
        tiles = blk.view(side, ps, n // side, ps, 3).permute(0, 2, 1, 3, 4).contiguous().view(n, ps, ps, 3)
        out['d_kernel_us_per_batch_7_levels'] = round(kernel_time(tiles, 7, args.kernel_reps), 2)
        out['d_batch_MB'] = round(tiles.numel() / 1e6, 2)
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
    if not all(same.values()):
        sys.exit('level files differ from compress_image of the reduction: %s' % same)


if __name__ == '__main__':
    main()
