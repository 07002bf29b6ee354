"""Region reads from a compressed slide: decode only the chunks a window touches.

With the reference, a compressed slide is a zarr array whose ``'cae'`` codec is registered with
numcodecs, so ``zarr.open(path)['0/0'][y0:y1, x0:x1]`` decodes the chunks under the window one
at a time through the codec (batch-1 synthesis, host coder, a host copy per chunk).  A slide is
compressed once and read many times, a window at a time: by a viewer, or by a patch sampler.

``CompressedSlide`` serves those reads without zarr.  Per call it plans the distinct chunks the
requested boxes touch (``plan``), reads their files with native threads, entropy-decodes all of
their streams in one device coder call (few streams go to the host coder on a thread pool), runs
the synthesis transform over ``batch_tiles`` tiles at a time with the kernels of the whole-slide
engine, and after every batch one launch of ``cae_tiles_crop_u8`` cuts the boxes' pieces out of
the decoded tiles on the device.  The pixels are the ones ``decompress_image`` writes.
"""
import os
import struct
import threading
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

from . import _autoencoders as AE
from . import _cabi as C
from . import _slide
from ._entropy import decode_symbols
from ._store import DirArray, _paths_blob, native_read


def plan(shape, chunks, boxes, box_h, box_w):
    """The chunks that the ``box_h`` x ``box_w`` boxes at ``boxes`` (N x 2 top-left (y, x)) of an
    array of ``shape`` (Y, X, ...) stored in ``chunks`` (cy, cx, ...) touch.

    Returns ``(chunk_yx, pieces)``: the distinct chunks as an int64 K x 2 array of chunk indices in
    row-major order, and an int32 P x 8 table ``{k, b, sy, sx, dy, dx, h, w}`` sorted by ``k``:
    rows [sy, sy + h) x columns [sx, sx + w) of chunk ``chunk_yx[k]`` are rows [dy, dy + h) x
    columns [dx, dx + w) of box ``b``.  Pieces end at the array edge: the padding of edge chunks
    is never read.  Raises ``ValueError`` for a box that does not lie inside the array."""
    H, W = int(shape[0]), int(shape[1])
    cy, cx = int(chunks[0]), int(chunks[1])
    box_h, box_w = int(box_h), int(box_w)
    if box_h <= 0 or box_w <= 0:
        raise ValueError('box size must be positive, got %d x %d' % (box_h, box_w))
    if cy <= 0 or cx <= 0:
        raise ValueError('chunk size must be positive')
    yx = np.asarray(boxes, dtype=np.int64).reshape(-1, 2)
    if len(yx) == 0:
        raise ValueError('no boxes')
    y, x = yx[:, 0], yx[:, 1]
    bad = (y < 0) | (x < 0) | (y + box_h > H) | (x + box_w > W)
    if bad.any():
        b = int(np.argmax(bad))
        raise ValueError('box %d (%d, %d) + %d x %d does not lie inside the %d x %d array'
                         % (b, y[b], x[b], box_h, box_w, H, W))
    gx = -(-W // cx)
    iy0, ix0 = y // cy, x // cx
    ny = (y + box_h - 1) // cy - iy0 + 1
    nx = (x + box_w - 1) // cx - ix0 + 1
    parts = []
    for a in range(int(ny.max())):
        for c in range(int(nx.max())):
            sel = np.nonzero((ny > a) & (nx > c))[0]
            iy, ix = iy0[sel] + a, ix0[sel] + c
            top = np.maximum(y[sel], iy * cy)
            left = np.maximum(x[sel], ix * cx)
            bottom = np.minimum(y[sel] + box_h, (iy + 1) * cy)
            right = np.minimum(x[sel] + box_w, (ix + 1) * cx)
            parts.append(np.stack([iy * gx + ix, sel, top - iy * cy, left - ix * cx,
                                   top - y[sel], left - x[sel], bottom - top, right - left], 1))
    pieces = np.concatenate(parts)
    ids, k = np.unique(pieces[:, 0], return_inverse=True)
    order = np.lexsort((pieces[:, 5], pieces[:, 4], pieces[:, 1], k))
    pieces[:, 0] = k
    chunk_yx = np.stack([ids // gx, ids % gx], 1)
    return chunk_yx, np.ascontiguousarray(pieces[order], dtype=np.int32)


def _index(key, n, axis):
    """(start, stop, keeps_axis) of one zarr-style basic index along an axis of length ``n``."""
    if isinstance(key, (int, np.integer)) and not isinstance(key, (bool, np.bool_)):
        k = int(key)
        if k < -n or k >= n:
            raise IndexError('index %d is out of bounds for axis %d with size %d' % (k, axis, n))
        k %= n
        return k, k + 1, False
    if isinstance(key, slice):
        if key.step not in (None, 1):
            raise IndexError('only slices with step 1 are supported (axis %d)' % axis)
        start, stop, _ = key.indices(n)
        return start, max(start, stop), True
    raise IndexError('unsupported index %r on axis %d: integers or step-1 slices only' % (key, axis))


class CompressedSlide:
    """Random access to the pixels of a ``'cae'`` array written by ``compress_image``.

    ``path``: the store; ``data_group``: the array inside it; ``checkpoint``: the model it was
    compressed with (a path or a state dict); ``batch_tiles``: tiles per synthesis batch (the
    full batches replay a CUDA graph); ``workers``: native I/O and host coder threads.

    The reader owns its model and its device buffers, so it can run beside ``decompress_image``
    calls on other threads; calls on one reader are serialised.  The decode graphs are captured
    when the reader is opened."""

    def __init__(self, path, checkpoint, data_group='0/0', batch_tiles=16, workers=None):
        from .compress import default_workers
        if not torch.cuda.is_available():
            raise RuntimeError('CompressedSlide needs a CUDA device (no CPU fallback)')
        self._arr = DirArray(os.path.join(path, data_group) if data_group else path, mode='r')
        codec_id = (self._arr.compressor_config or {}).get('id')
        if codec_id == 'cae_bn':
            raise ValueError("the array stores latents ('cae_bn'): its chunks are not pixels; "
                             "reconstruct the slide with decompress_image")
        if codec_id != 'cae':
            raise ValueError("array compressor %r is not the 'cae' codec" % codec_id)
        self.shape, self.chunks, self.dtype = self._arr.shape, self._arr.chunks, self._arr.dtype
        if len(self.shape) != 3 or self.dtype != np.uint8 or self.chunks[0] != self.chunks[1]:
            raise ValueError('expected a Y x X x C uint8 array in square chunks, got shape %r, '
                             'chunks %r, dtype %s' % (self.shape, self.chunks, self.dtype))
        self.ps = int(self.chunks[0])
        model = AE.autoencoder_from_state_dict(checkpoint, gpu=True, train=False)
        level = len(model['decoder'].module.synthesis_track)
        if self.ps % 2 ** level:
            raise ValueError('patch size %d is not a multiple of 2^%d' % (self.ps, level))
        last = model['decoder'].module.synthesis_track[-1]
        c_img = last.model[-1].out_channels if hasattr(last, 'model') else 3
        if c_img != self.shape[2]:
            raise ValueError('the model reconstructs %d channels, the array has %d'
                             % (c_img, self.shape[2]))
        self.model = model
        self.fact_ent = model['fact_ent'].module
        self.workers = workers or default_workers()
        self.tc = _slide.TileCodec(model, self.ps, c_img, int(batch_tiles),
                                   graphs=not os.environ.get('CAE_SLIDE_NO_GRAPHS'))
        self.tc.warm(encode=False, decode=True)
        self._tables = self.fact_ent._host_tables()
        self._pool = None
        self._pieces_dev = None
        self._uploaded = None             # the last upload out of the page-locked stream buffer
        self._lock = threading.Lock()
        self.stats = {}

    # ---- public reads ----
    def read_regions(self, boxes, h, w, out=None):
        """The ``h`` x ``w`` windows with top-left corners ``boxes`` ((y, x) pairs) as an
        N x h x w x c uint8 CUDA tensor (or in ``out``: a CUDA tensor, or a host ndarray --
        page-locked ones take an asynchronous copy; the call returns once it has landed)."""
        yx = np.asarray(boxes, dtype=np.int64).reshape(-1, 2)
        return self._read(yx, int(h), int(w), out, (len(yx), int(h), int(w), self.shape[2]))

    def read_region(self, y, x, h, w, out=None):
        """One ``h`` x ``w`` x c window at (y, x); ``out`` as for ``read_regions``."""
        return self._read(np.array([[y, x]], dtype=np.int64), int(h), int(w), out,
                          (int(h), int(w), self.shape[2]))

    def __getitem__(self, key):
        """zarr-style basic indexing on Y and X (integers, step-1 slices): a host ndarray."""
        key = key if isinstance(key, tuple) else (key,)
        if len(key) > 3 or (len(key) == 3 and key[2] != slice(None)):
            raise IndexError('only Y and X can be indexed (the channel axis is read whole)')
        key = tuple(key) + (slice(None),) * (2 - min(len(key), 2))
        y0, y1, keep_y = _index(key[0], self.shape[0], 0)
        x0, x1, keep_x = _index(key[1], self.shape[1], 1)
        out = np.empty((y1 - y0, x1 - x0, self.shape[2]), dtype=np.uint8)
        if out.size:
            self.read_region(y0, x0, y1 - y0, x1 - x0, out=out)
        return out[(slice(None) if keep_y else 0, slice(None) if keep_x else 0)]

    def close(self):
        if self._pool is not None:
            self._pool.shutdown()
            self._pool = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- the work ----
    def _read(self, yx, h, w, out, shape):
        chunk_yx, pieces = plan(self.shape, self.chunks, yx, h, w)
        dev = self.tc.dev
        host_out = None
        if out is None:
            dst = torch.empty(shape, dtype=torch.uint8, device=dev)
        elif isinstance(out, torch.Tensor):
            if (tuple(out.shape) != shape or out.dtype != torch.uint8 or out.device != dev
                    or not out.is_contiguous()):
                raise ValueError('out must be a contiguous uint8 tensor of shape %r on %s'
                                 % (shape, dev))
            dst = out
        elif isinstance(out, np.ndarray):
            if out.shape != shape or out.dtype != np.uint8 or not out.flags.c_contiguous:
                raise ValueError('out must be a C-contiguous uint8 ndarray of shape %r' % (shape,))
            host_out = out
            dst = torch.empty(shape, dtype=torch.uint8, device=dev)
        else:
            raise TypeError('out must be a CUDA tensor or a host ndarray')
        with self._lock, torch.cuda.device(dev):
            self._decode_and_crop(chunk_yx, pieces, dst, len(yx), h, w)
            if host_out is None:
                return dst
            if _slide.is_pinned_array(host_out):
                torch.from_numpy(host_out).copy_(dst, non_blocking=True)
                torch.cuda.current_stream(dev).synchronize()
            else:
                torch.from_numpy(host_out).copy_(dst)
            return host_out

    def _crop(self, tiles, n_tiles, pieces, dst, n_boxes, h, w):
        """One ``cae_tiles_crop_u8`` launch on the current stream (the piece table goes up on
        the same stream, so one device table serves every launch)."""
        if self._pieces_dev is None or self._pieces_dev.numel() < 8 * len(pieces):
            self._pieces_dev = torch.empty(8 * max(1024, len(pieces)), dtype=torch.int32,
                                           device=self.tc.dev)
        pieces = np.ascontiguousarray(pieces, dtype=np.int32)
        C.check(C.lib().cae_tiles_crop_u8(
            tiles.data_ptr() if tiles is not None else None, n_tiles, self.ps, self.tc.c_img,
            pieces.ctypes.data, len(pieces), self._pieces_dev.data_ptr(), dst.data_ptr(),
            n_boxes, h, w, _slide._stream_ptr(torch.cuda.current_stream(self.tc.dev))))

    def _decode_and_crop(self, chunk_yx, pieces, dst, n_boxes, h, w):
        """Decode the chunks ``chunk_yx`` group by group (``_slide.group_sizes``: the symbols of
        at most one group are on the device) and crop ``pieces`` out of every synthesis batch
        into ``dst``, on the current stream.  Returns once the device is done."""
        tc, fe, ps = self.tc, self.fact_ent, self.ps
        B, dev = tc.batch, tc.dev
        main = torch.cuda.current_stream(dev)
        paths = [self._arr.chunk_file((int(i), int(j), 0)) for i, j in chunk_yx]
        sizes = np.empty(len(paths), dtype=np.int64)
        C.check(C.lib().cae_files_stat(_paths_blob(paths), len(paths), sizes.ctypes.data,
                                       self.workers))
        present = sizes >= 0                   # a missing chunk file reads as the fill value 0
        # position of every chunk among the decoded ones (-1: missing), per piece
        piece_tile = np.where(present, np.cumsum(present) - 1, -1)[pieces[:, 0]]
        if not present.all():
            fill = pieces[piece_tile < 0].copy()
            fill[:, 0] = -1
            self._crop(None, 0, fill, dst, n_boxes, h, w)
        todo = [paths[k] for k in np.nonzero(present)[0]]
        self.stats = st = dict(chunks=len(paths), decoded=0, device_decoded=0,
                               missing=len(paths) - len(todo))
        expect_hdr = struct.pack('>QQ', ps, ps)
        statuses = []
        slot = lo = 0
        groups = _slide.group_sizes(len(todo), _slide.default_schedule(len(todo), B, decode=True),
                                    B) if todo else []
        for gn in groups:
            if self._uploaded is not None:
                self._uploaded.synchronize()  # the page-locked buffer's last upload has left it
            hdr, payload, off = native_read(todo[lo:lo + gn], 16, self.workers,
                                            alloc=lambda n: tc.pinned('region_streams', n).numpy())
            if bytes(hdr[0]) != expect_hdr or (hdr != hdr[0]).any():
                raise C.CaeError('chunk headers differ from the (patch, patch) the codec wrote')
            if gn >= fe.GPU_CODER_MIN_STREAMS:
                if (off % 4).any():
                    raise C.CaeError('chunk streams are not whole words')
                words = torch.empty(int(off[-1]) // 4, dtype=torch.int32, device=dev)
                words.view(torch.uint8).copy_(torch.from_numpy(payload), non_blocking=True)
                sym, status = fe.decode_streams_device(words, off // 4, tc.lh * tc.lw,
                                                       defer_status=True)
                statuses.append(status)
                st['device_decoded'] += gn
            else:
                # few streams: one host thread per stream beats the device coder's fixed cost
                if self._pool is None:
                    self._pool = ThreadPoolExecutor(max_workers=self.workers)
                cdf, sz, offs = self._tables
                sym = np.stack(list(self._pool.map(
                    lambda k: decode_symbols(payload[off[k]:off[k + 1]], tc.cb, tc.lh * tc.lw,
                                             cdf, sz, offs), range(gn))))
                sym = torch.from_numpy(sym).pin_memory().to(dev, non_blocking=True)
            self._uploaded = torch.cuda.Event()
            self._uploaded.record(main)
            sym = sym.reshape(gn, tc.cb, tc.lh, tc.lw)
            for p0 in range(0, gn, B):
                n = min(B, gn - p0)
                if n == B and tc.graphs:
                    tc.sym_in[slot].copy_(sym[p0:p0 + n], non_blocking=True)
                    u8 = tc.decode(slot, n)
                    slot = (slot + 1) % tc.slots
                else:
                    u8 = tc.decode_eager(sym[p0:p0 + n])
                t0 = lo + p0
                sel = (piece_tile >= t0) & (piece_tile < t0 + n)
                part = pieces[sel]
                part[:, 0] = piece_tile[sel] - t0
                self._crop(u8, n, part, dst, n_boxes, h, w)
            st['decoded'] += gn
            lo += gn
        main.synchronize()
        for status in statuses:
            fe.check_decode_status(status)
