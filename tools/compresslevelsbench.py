"""Pyramid levels at compression time (``compress_image(..., levels=K)``) at the bench size: the
slide, net and conventions of ``pyramidbench.py`` (8192 chunks of 512^2, 64 chunks per row, net A,
random-init seed 1234, ``batch_tiles`` 16).  For a pageable and for a page-locked source:

  (a) ``compress_image``;
  (b) ``compress_image(levels=7)``;
  (c) ``compress_image`` followed by ``CompressedSlide(...).build_pyramid()``: the route without
      compress-time levels.

Every call ends in a device synchronise.  After one warm-up call of each, (a), (b) and (c) are
called in turn, ``--calls`` rounds, so that a slow spell of the host falls on all three; every
call's time and peak device memory above its start are recorded, with the medians.  Level 0 of (b) is byte-compared with (a), and
every level of (b) with ``compress_image`` of the exact reduction of the source (block means
rounded half up, computed on the device in strips of chunk rows).  The PSNR of each level of (b)
and of (c) against that reduction is reported.  Prints one JSON line with the card name and
power limit.  The stores are written to ``/dev/shm`` when it has room, as ``bench.py`` does.

    python tools/compresslevelsbench.py [--chunks 8192] [--calls 3] [--out r.json]
"""
import argparse
import json
import os
import shutil
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import cae_oracle as O  # noqa: E402  (synthetic tiles + random-init checkpoint only)
from cnn_autoencoder_b200 import compress, decompress  # noqa: E402
from cnn_autoencoder_b200.region import CompressedSlide, level_shape  # noqa: E402
from tools.regionbench import card  # noqa: E402
from tools.regionreducebench import measure, summary  # noqa: E402


def files(d):
    return {f: open(os.path.join(d, f), 'rb').read() for f in sorted(os.listdir(d))}


def exact_levels(slide, levels, ps):
    """k -> the level-2^k image of ``slide`` (host uint8), reduced on the device one strip of ps
    rows at a time (every block is whole: the slide is made of whole chunks)."""
    H, W, c = slide.shape
    out = {k: np.empty(level_shape(slide.shape, 2 ** k), dtype=np.uint8) for k in range(1, levels + 1)}
    for y0 in range(0, H, ps):
        strip = torch.from_numpy(slide[y0:y0 + ps]).cuda().to(torch.int32)
        for k in range(1, levels + 1):
            f = 2 ** k
            s = strip.view(ps // f, f, W // f, f, c).sum(dim=(1, 3))
            n = f * f
            out[k][y0 // f:(y0 + ps) // f] = ((s + n // 2) // n).to(torch.uint8).cpu().numpy()
    return out


def psnr(a, b):
    mse = float(np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2))
    return round(10 * np.log10(255.0 ** 2 / mse), 3) if mse else float('inf')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--chunks', type=int, default=8192)
    ap.add_argument('--gx', type=int, default=64, help='chunks per row')
    ap.add_argument('--ps', type=int, default=512)
    ap.add_argument('--arch', default='A')
    ap.add_argument('--batch-tiles', type=int, default=16)
    ap.add_argument('--levels', type=int, default=7)
    ap.add_argument('--calls', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    ps, gx, K, B = args.ps, args.gx, args.levels, args.batch_tiles
    gy = -(-args.chunks // gx)
    H, W = gy * ps, gx * ps
    bank = {(i, j): O.synth_tissue_tile(i, j, ps=ps, seed=3) for i in range(4) for j in range(4)}
    pageable = np.empty((H, W, 3), dtype=np.uint8)
    for i in range(gy):
        for j in range(gx):
            pageable[i * ps:(i + 1) * ps, j * ps:(j + 1) * ps] = bank[(i % 4, j % 4)]
    chk = O.make_checkpoint(O.NAMED_ARCHS[args.arch], seed=1234)
    out = dict(card=None, power_limit=None, arch=args.arch, chunks=gy * gx, ps=ps, slide_px=[H, W],
               levels=K, batch_tiles=B, calls=args.calls)
    out['card'], out['power_limit'] = card()
    # the stores go to tmpfs where there is room, as bench.py's: every call writes 1.1-1.5 GB of
    # chunk files, and on a disk-backed /tmp their writeback throttles some calls, not others
    shm = os.path.isdir('/dev/shm') and shutil.disk_usage('/dev/shm').free > 3 * H * W
    base = tempfile.mkdtemp(prefix='compresslevelsbench_', dir='/dev/shm' if shm else None)
    out['store'] = 'tmpfs' if shm else tempfile.gettempdir()
    same = {}
    try:
        exact = exact_levels(pageable, K, ps)
        ref = {}
        for k in range(1, K + 1):
            p = os.path.join(base, 'ref%d.zarr' % k)
            compress.compress_image('CAE', chk, exact[k], p, patch_size=ps, batch_tiles=B)
            ref[k] = files(os.path.join(p, '0', '0'))
            shutil.rmtree(p)
        pinned = torch.from_numpy(pageable).pin_memory().numpy()
        for kind, src in (('pageable', pageable), ('pinned', pinned)):
            pa, pb, pc = (os.path.join(base, '%s_%s.zarr' % (kind, r)) for r in 'abc')
            st, reader = {}, []

            def a(_):
                st['a'] = compress.compress_image('CAE', chk, src, pa, patch_size=ps, batch_tiles=B)

            def b(_):
                st['b'] = compress.compress_image('CAE', chk, src, pb, patch_size=ps, batch_tiles=B,
                                                  levels=K)

            def c(_):
                compress.compress_image('CAE', chk, src, pc, patch_size=ps, batch_tiles=B)
                if not reader:           # opened once (model, graphs), outside the timed calls
                    reader.append(CompressedSlide(pc, chk, mode='r+', batch_tiles=B))
                reader[0].build_pyramid(levels=K, overwrite=True)
            routes = (('a_compress', a), ('b_compress_levels%d' % K, b),
                      ('c_compress_then_build_pyramid', c))
            for _, fn in routes:
                fn(None)                                        # warm-up
            calls = {name: ([], []) for name, _ in routes}
            for r in range(args.calls):                         # alternated, call by call
                for name, fn in routes:
                    t, p = measure(fn, [r])
                    calls[name][0].append(t[0])
                    calls[name][1].append(p[0])
            for name, (t, p) in calls.items():
                out['%s_%s' % (kind, name)] = summary(
                    t, p, s_median=round(float(np.median(t)), 3), s_calls=[round(x, 3) for x in t],
                    peak_MB_calls=[round(x / 2 ** 20, 1) for x in p])
            med = {name[0]: out['%s_%s' % (kind, name)]['s_median'] for name, _ in routes}
            out['%s_b_minus_a_s' % kind] = round(med['b'] - med['a'], 3)
            out['%s_c_minus_b_s' % kind] = round(med['c'] - med['b'], 3)
            # per round: the three calls ran back to back
            out['%s_b_minus_a_s_per_round' % kind] = [
                round(x - y, 3) for x, y in zip(*(calls[name][0] for name, _ in routes[1::-1]))]
            out['%s_b_stats' % kind] = {k: st['b'][k] for k in ('bytes', 'level_chunks',
                                                                  'level_bytes', 'device_coded')}
            same['%s_level0_b_equals_a' % kind] = files(os.path.join(pa, '0', '0')) == \
                files(os.path.join(pb, '0', '0'))
            for k in range(1, K + 1):
                same['%s_level%d_b_equals_reference' % (kind, k)] = \
                    files(os.path.join(pb, '0', str(k))) == ref[k]
            if kind == 'pageable':
                for r, path in (('b', pb), ('c', pc)):
                    out['psnr_%s' % r] = {}
                    for k in range(1, K + 1):
                        img = torch.zeros(exact[k].shape, dtype=torch.uint8).pin_memory().numpy()
                        decompress.decompress_image(path, img, data_group='0/%d' % k,
                                                    checkpoint=chk, batch_tiles=B)
                        out['psnr_%s' % r][k] = psnr(img, exact[k])
            reader[0].close()
            for d in (pa, pb, pc):
                shutil.rmtree(d)
        out['outputs_equal'] = same
    finally:
        shutil.rmtree(base, ignore_errors=True)
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')
    if not all(same.values()):
        sys.exit('level files differ: %s' % same)


if __name__ == '__main__':
    main()
