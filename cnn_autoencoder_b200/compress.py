"""Whole-slide compression tile loop, mirroring ``src/compress.py`` of the
reference (``compress_image`` :29-168, ``compress`` :171-209) for the CAE codecs.

The reference hands every ``patch_size`` chunk to the codec one at a time from
dask's threaded scheduler (``z.rechunk(...)`` :101, ``to_zarr(compressor=codec)``
:121-128).  Here the same chunks are processed B200-first: native threads cut
``batch_tiles`` tiles out of the slide into a pinned buffer, the analysis transform +
quantizer run once per batch on the GPU, and the integer symbols of up to ``coder_tiles``
tiles stay on the device, where every tile's rANS stream is coded concurrently on a second
CUDA stream while the transforms of the next tiles run; the packed streams come back in one
copy and native threads write the chunk files.  (Below 128 tiles per call the C++ host
coder, on a thread pool, is faster and is used instead.)
Tiles are independent (no halo between chunks), so ``world_size`` processes -- one
per GPU -- each take a contiguous range of the chunk grid and write their own chunk
files; there is no collective.  The output is a zarr-v2 directory array whose
compressor entry is the codec config, chunk for chunk what the reference writes.
"""
import argparse
import math
import os
import struct
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

from . import _autoencoders as AE
from ._entropy import encode_symbols
from . import _slide
from . import region
from ._store import DirArray, can_native_gather, native_gather, native_write, padded_tile

_models = {}


def load_model(checkpoint):
    """``autoencoder_from_state_dict(checkpoint, gpu=True, train=False)`` (R:505-527), kept for
    the next call on the same checkpoint: a slide is usually one of many compressed with one
    model, and the packed weights / CUDA graphs hang off the model objects."""
    if isinstance(checkpoint, str):
        key = ('path', checkpoint, os.path.getmtime(checkpoint), torch.cuda.current_device())
    else:
        # (the three table buffers of fact_ent are shared with the module while loading and
        # rewritten by update(): not part of the identity of a checkpoint)
        sig = tuple((k, v.data_ptr(), v._version) for part in ('encoder', 'decoder', 'fact_ent')
                    for k, v in sorted((checkpoint.get(part) or {}).items())
                    if k not in ('_quantized_cdf', '_offset', '_cdf_length'))
        key = ('dict', id(checkpoint), hash(sig), torch.cuda.current_device())
    m = _models.get(key)
    if m is None:
        if len(_models) >= 4:
            _models.clear()
        m = _models[key] = AE.autoencoder_from_state_dict(checkpoint=checkpoint, gpu=True,
                                                          train=False)
    return m


def shard_range(n_items, rank, world_size):
    """Contiguous chunk range [k*n/G, (k+1)*n/G) of rank k (SURVEY.md 8d-4, 8e)."""
    return range(rank * n_items // world_size, (rank + 1) * n_items // world_size)


def _dist_info(rank, world_size):
    if rank is None:
        rank = int(os.environ.get('RANK', 0))
    if world_size is None:
        world_size = int(os.environ.get('WORLD_SIZE', 1))
    return rank, world_size


def default_workers():
    """Native I/O threads of one rank: the host cores are shared by the ranks of the box
    (torchrun exports LOCAL_WORLD_SIZE), oversubscribing them slows every rank."""
    local = max(1, int(os.environ.get('LOCAL_WORLD_SIZE', 1)))
    return max(2, min(32, (os.cpu_count() or 4) // local))


def open_source(input_filename, data_group='0/0'):
    """H x W x C uint8 array-like from: an ndarray, a ``.npy`` path (memory mapped), a
    directory array written by ``_store.DirArray`` (``<path>/<data_group>``), or -- when
    the optional ``zarr`` package is installed -- any zarr v2 array."""
    if isinstance(input_filename, np.ndarray):
        return input_filename
    if input_filename.endswith('.npy'):
        return np.load(input_filename, mmap_mode='r')
    path = os.path.join(input_filename, data_group) if data_group else input_filename
    try:
        import zarr                                    # optional
        return zarr.open(input_filename, mode='r')[data_group]
    except ImportError:
        pass
    arr = DirArray(path, mode='r')
    if arr.compressor_config is not None:
        raise ValueError('source array is compressed; only raw directory arrays can be read '
                         'without the zarr package')

    class _View:
        shape, dtype = arr.shape, arr.dtype

        def __getitem__(self, key):
            ys, xs = key[0], key[1]
            out = np.empty((ys.stop - ys.start, xs.stop - xs.start, arr.shape[2]), arr.dtype)
            cy, cx = arr.chunks[0], arr.chunks[1]
            for iy in range(ys.start // cy, -(-ys.stop // cy)):
                for ix in range(xs.start // cx, -(-xs.stop // cx)):
                    blk = arr.read_chunk((iy, ix, 0))
                    y0, x0 = iy * cy, ix * cx
                    a, b = max(ys.start, y0), min(ys.stop, y0 + blk.shape[0])
                    c, d = max(xs.start, x0), min(xs.stop, x0 + blk.shape[1])
                    out[a - ys.start:b - ys.start, c - xs.start:d - xs.start] = \
                        blk[a - y0:b - y0, c - x0:d - x0]
            return out

    return _View()


class _AxesView:
    """Y x X x C view of an array stored with other axes (``compress.py:89-101`` of the
    reference: transpose to <other axes> + YXC and take index 0 of every other axis)."""

    def __init__(self, arr, axes):
        self.arr, self.axes = arr, axes
        pos = {a: i for i, a in enumerate(axes)}
        self.shape = (arr.shape[pos['Y']], arr.shape[pos['X']], arr.shape[pos['C']])
        self.dtype = arr.dtype
        self.pos = pos

    def __getitem__(self, key):
        key = key if isinstance(key, tuple) else (key,)
        key = tuple(key) + (slice(None),) * (3 - len(key))
        index = [0] * len(self.axes)
        for a, k in zip('YXC', key):
            index[self.pos[a]] = k
        block = np.asarray(self.arr[tuple(index)])
        kept = [a for a in self.axes if a in 'YXC' and not isinstance(index[self.pos[a]], int)]
        return np.ascontiguousarray(block.transpose([kept.index(a) for a in 'YXC' if a in kept]))


def as_yxc(src, data_axes):
    """The source as an H x W x C array-like.  Arrays that already are three-dimensional are
    taken as YXC whatever ``data_axes`` says (the ndarray / ``.npy`` / directory-array sources of
    this package); anything else is mapped like the reference does."""
    shape = tuple(src.shape)
    if len(shape) == 3:
        return src
    axes = str(data_axes).upper()
    if len(axes) != len(shape) or not set('YXC') <= set(axes) or len(set(axes)) != len(axes):
        raise ValueError('source has shape %r, which data_axes=%r does not describe (need one '
                         'letter per axis including Y, X and C)' % (shape, data_axes))
    return _AxesView(src, axes)


def check_levels(levels, shape, ps, save_as_bottleneck=False, world_size=1, data_group='0/0'):
    """The number K of pyramid levels ``compress_image(..., levels=levels)`` writes for a
    Y x X x c source in ps^2 chunks (0: none).  ``levels``: 0, K >= 1 (``region.check_levels``) or
    ``'auto'`` (``region.default_levels``).  Raises ``ValueError`` for a bad K, and for levels with
    ``save_as_bottleneck``, ``world_size > 1`` or a data group whose last component is not ``0``."""
    if isinstance(levels, str):
        if levels != 'auto':
            raise ValueError("levels must be an int or 'auto', got %r" % (levels,))
        K = region.default_levels(shape, ps)
    elif isinstance(levels, (int, np.integer)) and not isinstance(levels, (bool, np.bool_)) \
            and int(levels) == 0:
        return 0
    else:
        K = region.check_levels(levels, ps)
    if save_as_bottleneck:
        raise ValueError('levels: a latent store (save_as_bottleneck) has no pixel levels')
    if world_size > 1:
        raise ValueError('levels: the shards of a sharded job are contiguous tile ranges that split '
                         'chunk rows; compress without levels, then run '
                         "CompressedSlide(path, checkpoint, mode='r+').build_pyramid()")
    if region.pyramid_group('', data_group) is None:
        raise ValueError("levels go beside a '<group>/0' array; the data group is %r" % (data_group,))
    return K


def compress_image(codec, checkpoint, input_filename, output_filename, patch_size=512,
                   source_format='zarr', data_group='0/0', data_axes='TCZYX',
                   progress_bar=False, save_as_bottleneck=False, gpu=False, *,
                   rank=None, world_size=None, batch_tiles=16, workers=None, coder_tiles=None,
                   levels=0):
    """Same positional signature as the reference (``compress.py:29-36``); the keyword-only
    arguments select this process's shard, the GPU batch size and how many tiles are entropy
    coded per device call (one size, or a schedule of group sizes: ``_slide.group_sizes``).  Returns a dict of counters (tiles, pixels, bytes, seconds,
    device_coded) for the caller's throughput report.

    ``levels``: also write the resolution pyramid in the same pass (0: no, the default; K: levels
    1..K; ``'auto'``: ``region.default_levels``; see ``check_levels``).  Level k is the ``'cae'``
    array ``<group>/k`` beside ``<group>/0``, with the same codec config and chunks; its files are
    the ones this function writes for ``reduce(source, 2^k)``, the block means of the *source*
    rounded half up (edge blocks average the pixels inside the array), and ``<group>/.zattrs``
    gets the ``multiscales`` entry of ``CompressedSlide.build_pyramid``.  This is the one
    difference from ``build_pyramid``, whose levels are means of the decoded slide: levels
    written here carry one lossy encode, not two.  Every uploaded batch is reduced into one
    chunk row per level on the device (``region.PyramidWriter``); nothing is decoded.  An
    existing entry is removed before any chunk is written and the new one is written last, so a
    failed call leaves no entry listing incomplete levels; the chunks of levels 1..K are removed
    like level 0's, and stored levels above K are left in place, unlisted.  The stats gain
    ``level_chunks`` and ``level_bytes``; ``bytes``, ``tiles`` and ``pixels`` count level 0."""
    if 'CAE' not in codec:
        raise ValueError('Codec %s not supported' % codec)
    if not torch.cuda.is_available():
        raise RuntimeError('compress_image needs a CUDA device (no CPU fallback)')
    rank, world_size = _dist_info(rank, world_size)
    workers = workers or default_workers()
    src = as_yxc(open_source(input_filename, data_group), data_axes)
    H, W, C = src.shape
    ps = patch_size
    K = check_levels(levels, (H, W, C), ps, save_as_bottleneck, world_size, data_group)

    model = load_model(checkpoint)
    fact_ent = model['fact_ent'].module
    channels_bn = fact_ent.channels
    level = len(model['encoder'].module.analysis_track)
    cdf, sizes, offs = fact_ent._host_tables()

    gy, gx = -(-H // ps), -(-W // ps)
    out_path = os.path.join(output_filename, data_group) if data_group else output_filename
    if save_as_bottleneck:
        # '-sbn': the stored array is the latent; chunks ceil(cs / 2^L) (compress.py:103-109).
        # The reference runs the analysis transform on the edge tiles at their true size
        # (map_blocks, :111-113); the stride-2 kernels here need even sizes at every level, so a
        # slide whose edge tiles are not multiples of 2^L is refused before any work is done.
        for name, size in (('height', H), ('width', W)):
            edge = size % ps
            if edge % (2 ** level):
                raise ValueError('save_as_bottleneck: the edge tiles of this slide are %d px in %s, '
                                 'not a multiple of 2^%d; pad or crop the slide' % (edge, name, level))
        comp = AE.ConvolutionalAutoencoderBottleneck(channels_bn=channels_bn, fact_ent=fact_ent,
                                                     gpu=True)
        lat = lambda v: int(math.ceil(v / 2 ** level))
        shape = (sum(lat(min(ps, H - i * ps)) for i in range(gy)),
                 sum(lat(min(ps, W - j * ps)) for j in range(gx)), channels_bn)
        meta = dict(shape=shape, chunks=(lat(ps), lat(ps), channels_bn), dtype=np.float32)
    else:
        comp = _CodecConfig('cae', checkpoint=checkpoint if isinstance(checkpoint, str) else '<dict>',
                            gpu=gpu)
        meta = dict(shape=(H, W, C), chunks=(ps, ps, C), dtype=np.uint8)
    level_arrays = []
    if K:
        group = region.pyramid_group(output_filename, data_group)
        if 'multiscales' in region._read_attrs(group):
            region.write_multiscales(output_filename, group, 0)
    if rank == 0:
        dst = DirArray(out_path, compressor=comp, mode='w', **meta)
        if world_size == 1:
            # overwrite=True of the reference's to_zarr (compress.py:123-128): the chunks of an
            # array that was there before are gone.  The ranks of a sharded job have no barrier
            # between this and the first chunk another rank writes, so there stale chunks stay.
            dst.remove_chunks(workers)
        for k in range(1, K + 1):
            level_arrays.append(DirArray(os.path.join(group, str(k)), compressor=comp, mode='w',
                                         shape=region.level_shape((H, W, C), 2 ** k),
                                         chunks=(ps, ps, C), dtype=np.uint8))
            level_arrays[-1].remove_chunks(workers)
    else:
        while not os.path.exists(os.path.join(out_path, '.zarray')):
            time.sleep(0.05)
        dst = DirArray(out_path, mode='r')

    tiles = [(i, j) for i in range(gy) for j in range(gx)]
    mine = [tiles[k] for k in shard_range(len(tiles), rank, world_size)]
    if coder_tiles is None:
        coder_tiles = _slide.default_schedule(len(mine), batch_tiles, decode=False)
    stats = dict(tiles=len(mine), pixels=0, bytes=0, seconds=0.0, device_coded=0,
                 t_read=0.0, t_stage=0.0, t_gpu=0.0, t_code=0.0, t_write_wait=0.0)
    t_start = time.perf_counter()
    if (not save_as_bottleneck and can_native_gather(src) and ps % (2 ** level) == 0
            and len(mine) >= fact_ent.GPU_CODER_MIN_STREAMS and not os.environ.get('CAE_NO_SLIDE_ENGINE')):
        # the batched engine: strided DMA out of the slide, one CUDA-graph replay per batch, all
        # streams of a group coded on the device (see _slide.py)
        tc = _slide.tile_codec(model, ps, C, batch_tiles)
        if len(mine) >= batch_tiles:
            tc.warm(encode=True, decode=False, level=bool(K))
        t_start = time.perf_counter()
        st = _slide._Stats(want_trace=bool(os.environ.get('CAE_SLIDE_TRACE')))
        _slide.compress_tiles(tc, src, mine, dst.chunk_file, (ps, ps), workers, coder_tiles, st,
                              level_arrays=level_arrays)
        stats.update(st)
        stats['engine'] = 'slide'
        stats['seconds'] = time.perf_counter() - t_start
        if K:
            region.write_multiscales(output_filename, group, K)
        return stats
    if not isinstance(coder_tiles, (int, np.integer)):
        coder_tiles = max(int(g) for g in coder_tiles)     # a group schedule (_slide.group_sizes)
    pool = ThreadPoolExecutor(max_workers=workers)
    writes = []                     # futures of chunk-file writes
    acc = {}                        # latent shape -> dict(sym=[device tensors], meta=[(idx, h, w)])
    coder = ThreadPoolExecutor(max_workers=1)      # entropy-codes one group while the transforms
    coder_stream = torch.cuda.Stream()             # of the next group run on the main stream
    coder_jobs = []
    out_pin = [None]                               # reused pinned buffer of the coder thread

    def coder_pinned(n):
        # page-locked allocations stall every other CUDA call of the process: one buffer for
        # every group of the coder thread, only grown
        if out_pin[0] is None or out_pin[0].numel() < n:
            out_pin[0] = torch.empty(int(n * 1.25) + 4096, dtype=torch.uint8, pin_memory=True)
        return out_pin[0][:n]
    device = torch.cuda.current_device()

    def write_stream(idx, h, w, data):
        dst.write_encoded(idx, struct.pack('>QQ', h, w), data)
        return 16 + len(data)

    def flush_group(key, final=False):
        """Entropy-code the accumulated tiles of one latent shape.  With enough tiles in flight
        every stream is coded concurrently on the device (the symbols never visit the host);
        a small remainder goes to the host coder threads instead (one device call costs the
        same ~70 ms whatever the stream count)."""
        g = acc.pop(key, None)
        if not g or not g['meta']:
            return
        t0 = time.perf_counter()
        sym = g['sym'][0] if len(g['sym']) == 1 else torch.cat(g['sym'])
        n = sym.shape[0]
        if n >= fact_ent.GPU_CODER_MIN_STREAMS:
            ready = torch.cuda.Event()
            ready.record()                       # the symbols are complete at this point

            def job(sym=sym, meta=g['meta'], ready=ready):
                torch.cuda.set_device(device)
                with torch.cuda.stream(coder_stream):
                    coder_stream.wait_event(ready)
                    packed, off = fact_ent.encode_symbols_device(sym)
                    host = coder_pinned(packed.numel())
                    host.copy_(packed, non_blocking=True)
                    coder_stream.synchronize()
                # one native call writes the group's chunk files (16-byte header + stream each)
                hdr = np.frombuffer(b''.join(struct.pack('>QQ', h, w) for _, h, w in meta),
                                    dtype=np.uint8).reshape(len(meta), 16)
                native_write([dst.chunk_file(idx) for idx, _, _ in meta], hdr, host.numpy(), off,
                             workers)
                stats['bytes'] += int(off[-1]) + 16 * len(meta)
                return []
            coder_jobs.append(coder.submit(job))
            stats['device_coded'] += n
        else:
            sym_h = sym.reshape(n, sym.shape[1], -1).cpu().numpy()
            for k, (idx, h, w) in enumerate(g['meta']):
                writes.append(pool.submit(
                    lambda k=k, idx=idx, h=h, w=w: write_stream(
                        idx, h, w, encode_symbols(sym_h[k], cdf, sizes, offs))))
        stats['t_code'] += time.perf_counter() - t0

    def run_batch(batch):
        """batch: list of ((i, j), tile) with identical tile shapes; ``tile`` is an ndarray or
        None (full ps x ps chunk, read from the source straight into the staging buffer)."""
        th, tw = batch[0][1].shape[:2] if batch[0][1] is not None else (ps, ps)
        t0 = time.perf_counter()
        pin = _pinned((len(batch), th, tw, C))
        if id(pin) in staged:
            staged.pop(id(pin)).synchronize()          # its previous upload has been consumed
        pin_np = pin.numpy()
        if native_src and batch[0][1] is None:
            native_gather(src, ps, np.array([ij for ij, _ in batch], dtype=np.int32), pin_np, workers)
            batch_done = True
        else:
            batch_done = False

        def put(k):
            (i, j), tile = batch[k]
            if tile is not None:
                pin_np[k] = tile
                return
            y0, x0 = i * ps, j * ps
            part = src[y0:min(y0 + ps, H), x0:min(x0 + ps, W)]
            if part.shape[0] != ps or part.shape[1] != ps:
                pin_np[k] = 0                          # edge chunk: zero fill, as zarr pads
            pin_np[k, :part.shape[0], :part.shape[1]] = part
        if not batch_done:
            list(pool.map(put, range(len(batch))))
        x = pin.cuda(non_blocking=True)
        t1 = time.perf_counter()
        stats['t_stage'] += t1 - t0
        # stand-alone quantizer by default (see pipeline.CodecPipeline for the measurement)
        req = fact_ent.quant_request(want_sym=True, want_planar=False, want_yq=False,
                                     want_stats=False) if os.environ.get('CAE_FUSED_QUANT') else None
        y = model['encoder'](x, quant=req)
        if save_as_bottleneck and (y.shape[2] != lat(ps) or y.shape[3] != lat(ps)):
            # edge chunk of the latent array: zarr pads it to the full chunk with the fill value 0
            # before the codec sees it (compress.py:121-128 -> R:637-651), header = full chunk
            full = torch.zeros((y.shape[0], y.shape[1], lat(ps), lat(ps)), dtype=y.dtype, device=y.device)
            full[:, :, :y.shape[2], :y.shape[3]] = y
            y, req = full, None
        if req is not None and req.done:
            sym = req.sym                        # quantized in the last encoder layer's epilogue
        else:
            _, _, sym, _, _ = fact_ent._quantize_cuda(y, want_yq=False, want_p=False, want_sym=True)
        lh, lw = y.shape[2], y.shape[3]
        hh, ww = (lh, lw) if save_as_bottleneck else (th, tw)
        stats['pixels'] += len(batch) * th * tw
        if pyr is not None:
            pyr.add(x, [ij for ij, _ in batch])
        g = acc.setdefault((lh, lw), dict(sym=[], meta=[]))
        g['sym'].append(sym)
        g['meta'] += [((idx[0], idx[1], 0), hh, ww) for idx, _ in batch]
        staged[id(pin)] = torch.cuda.Event()
        staged[id(pin)].record()                       # the staging buffer is free after this
        stats['t_gpu'] += time.perf_counter() - t1
        if len(g['meta']) >= coder_tiles:
            flush_group((lh, lw))

    def load(ij):
        i, j = ij
        if save_as_bottleneck:
            return np.ascontiguousarray(src[i * ps:min((i + 1) * ps, H), j * ps:min((j + 1) * ps, W)])
        return padded_tile(src, i * ps, j * ps, ps)

    pinned, staged = {}, {}
    native_src = can_native_gather(src)      # in-memory / memory-mapped slide: native tile gather

    def _pinned(shape):
        # two reusable pinned staging buffers per batch shape, used alternately (page-locking
        # per batch is slow; alternating lets batch k+1 be staged while batch k uploads)
        ring = pinned.setdefault(shape, [])
        if len(ring) < 2:
            ring.append(torch.empty(shape, dtype=torch.uint8).pin_memory())
            return ring[-1]
        ring.append(ring.pop(0))
        return ring[-1]

    pyr = None
    if K:
        def level_group(sym, paths):
            ready = torch.cuda.Event()
            ready.record()

            def job():
                # through the coder thread, which serialises the device coder calls
                torch.cuda.set_device(device)
                with torch.cuda.stream(coder_stream):
                    coder_stream.wait_event(ready)
                    nbytes, _ = _slide.code_and_write(fact_ent, (cdf, sizes, offs), sym, paths, ps,
                                                      workers, coder_pinned, pool)
                stats['level_bytes'] += nbytes
                return []
            coder_jobs.append(coder.submit(job))

        # chunks come in row-major order: the batches are reduced as they are encoded
        pyr = region.PyramidWriter((H, W, C), ps, K, batch_tiles, device,
                                   lambda k, idx: level_arrays[k - 1].chunk_file(idx),
                                   lambda run: _slide.encode_tiles(model['encoder'], fact_ent, run),
                                   level_group, (channels_bn, (ps // 2 ** level) ** 2))
        stats.update(level_chunks=len(pyr.paths), level_bytes=0)

    groups = {}
    for k0 in range(0, len(mine), batch_tiles):
        part = mine[k0:k0 + batch_tiles]
        if not save_as_bottleneck:
            run_batch([(ij, None) for ij in part])            # one copy: source -> pinned buffer
            continue
        t0 = time.perf_counter()
        loaded = list(pool.map(load, part))                   # tile reads in parallel
        stats['t_read'] += time.perf_counter() - t0
        for ij, tile in zip(part, loaded):
            g = groups.setdefault(tile.shape, [])
            g.append((ij, tile))
            if len(g) == batch_tiles:
                run_batch(g)
                groups[tile.shape] = []
    for g in groups.values():
        if g:
            run_batch(g)
    for key in list(acc):
        flush_group(key, final=True)
    if pyr is not None:
        pyr.finish()
    t0 = time.perf_counter()
    for j in coder_jobs:
        writes += j.result()
    for f in writes:
        stats['bytes'] += f.result()
    stats['t_write_wait'] = time.perf_counter() - t0
    coder.shutdown()
    pool.shutdown()
    torch.cuda.synchronize()
    if K:
        region.write_multiscales(output_filename, group, K)
    stats['seconds'] = time.perf_counter() - t_start
    return stats


class _CodecConfig:
    """Carries the 'cae' codec config into ``.zarray`` without loading a second model."""

    def __init__(self, codec_id, **cfg):
        self.codec_id = codec_id
        self._cfg = cfg

    def get_config(self):
        return dict(id=self.codec_id, **self._cfg)


def compress(args):
    """CLI driver (``compress.py:171-209``): every input file -> ``<name>.zarr``."""
    inputs = args.data_dir if isinstance(args.data_dir, (list, tuple)) else [args.data_dir]
    for fn in inputs:
        if '.zarr' in args.output_dir.lower():
            out = args.output_dir
        else:
            base = os.path.basename(fn.rstrip('/')).split('.')[0]
            out = os.path.join(args.output_dir, base + '.zarr')
        st = compress_image(codec=args.codec, checkpoint=args.checkpoint, input_filename=fn,
                            output_filename=out, patch_size=args.patch_size,
                            data_group=args.data_group, save_as_bottleneck=args.save_as_bottleneck,
                            gpu=True, batch_tiles=args.batch_tiles, levels=args.levels)
        print('Compressed image %s into %s: %d tiles, %.1f MP/s' % (
            fn, out, st['tiles'], st['pixels'] / 1e6 / max(st['seconds'], 1e-9)))


def _parser():
    ap = argparse.ArgumentParser(description='B200 CAE whole-slide compression')
    ap.add_argument('-chk', '--checkpoint', required=True)
    ap.add_argument('-dd', '--data-dir', nargs='+', required=True)
    ap.add_argument('-o', '--output-dir', required=True)
    ap.add_argument('-ps', '--patch-size', type=int, default=512)
    ap.add_argument('-cod', '--codec', default='CAE')
    ap.add_argument('-dg', '--data-group', default='0/0')
    ap.add_argument('-sbn', '--save-as-bottleneck', action='store_true')
    ap.add_argument('-g', '--gpu', action='store_true')
    ap.add_argument('--batch-tiles', type=int, default=16)
    ap.add_argument('--levels', type=_levels_arg, default=0,
                    help="also write pyramid levels 1..K (an int, or 'auto'); off by default")
    return ap


def _levels_arg(text):
    if text == 'auto':
        return text
    try:
        return int(text)
    except ValueError:
        raise argparse.ArgumentTypeError("expected an int or 'auto', got %r" % text) from None


if __name__ == '__main__':
    compress(_parser().parse_args())
