"""Region reads from and writes to a compressed slide: code only the chunks a window touches.

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

``CompressedSlide.downsampled(f)`` (``SlideLevel``) reads the slide at 1/f of its resolution, as
a viewer or a 20x / 10x patch sampler wants it: the same decode, and after every batch one launch
of ``cae_tiles_crop_reduce_u8`` box-filters the pieces (``reduce_plan``) into the level image.

Opened with ``mode='r+'`` (or made empty by ``create_slide``) it also writes, as zarr's
assignment does: a read-modify-write per touched chunk.  ``write_plan`` adds to ``plan`` which
chunks are covered whole (encoded without reading them) and the zero pieces of edge padding; the
partly covered chunks are decoded as for a read, every batch of tiles is assembled on the device
with one ``cae_tiles_paste_u8`` launch, encoded with the engine's kernels, entropy-coded per
group and written as chunk files.  The padding of an edge chunk is always stored as zeros
(``compress_image`` does the same; zarr would keep the decoded padding), so writing a slide in
whole chunks gives ``compress_image``'s files byte for byte.
"""
import json
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


def check_disjoint(boxes, box_h, box_w):
    """Raise ``ValueError`` if two of the ``box_h`` x ``box_w`` boxes at ``boxes`` (N x 2 top-left
    (y, x)) share a pixel: a write of overlapping boxes would depend on their order."""
    yx = np.asarray(boxes, dtype=np.int64).reshape(-1, 2)
    order = np.lexsort((yx[:, 1], yx[:, 0]))
    y, x = yx[order, 0], yx[order, 1]
    # sorted by y: once no pair d apart is closer than box_h in y, no pair further apart is
    for d in range(1, len(y)):
        near = y[d:] - y[:-d] < box_h
        if not near.any():
            break
        hit = near & (np.abs(x[d:] - x[:-d]) < box_w)
        if hit.any():
            i = int(np.argmax(hit))
            a, b = sorted((int(order[i]), int(order[i + d])))
            raise ValueError('boxes %d and %d overlap: a write would depend on their order' % (a, b))


def write_plan(shape, chunks, boxes, box_h, box_w):
    """What a write of the ``box_h`` x ``box_w`` boxes at ``boxes`` needs: ``plan`` plus, per
    touched chunk, whether the boxes cover its whole in-array part, and the zero pieces of its
    padding.

    Returns ``(chunk_yx, pieces, full, fill)``: ``chunk_yx`` and ``pieces`` as ``plan`` returns
    them; ``full``: bool K, the chunks whose in-array part is covered (they are encoded without
    reading their old file); ``fill``: int32 F x 8 pieces ``{k, -1, sy, sx, 0, 0, h, w}`` covering
    the part of every touched edge chunk beyond the array edge (stored as zeros).  Value and fill
    pieces are pairwise disjoint.  Raises ``ValueError`` for overlapping boxes."""
    chunk_yx, pieces = plan(shape, chunks, boxes, box_h, box_w)
    check_disjoint(boxes, box_h, box_w)
    H, W = int(shape[0]), int(shape[1])
    cy, cx = int(chunks[0]), int(chunks[1])
    ih = np.minimum(cy, H - chunk_yx[:, 0] * cy)          # in-array rows / columns of each chunk
    iw = np.minimum(cx, W - chunk_yx[:, 1] * cx)
    covered = np.bincount(pieces[:, 0], weights=pieces[:, 6].astype(np.int64) * pieces[:, 7],
                          minlength=len(chunk_yx))
    full = covered == ih * iw                            # the boxes are disjoint: areas add up
    k = np.arange(len(chunk_yx))
    zero = np.zeros_like(k)
    below = np.stack([k, zero - 1, ih, zero, zero, zero, cy - ih, zero + cx], 1)[ih < cy]
    right = np.stack([k, zero - 1, zero, iw, zero, zero, ih, cx - iw], 1)[iw < cx]
    fill = np.concatenate([below, right])
    return chunk_yx, pieces, full, np.ascontiguousarray(fill[np.argsort(fill[:, 0], kind='stable')],
                                                        dtype=np.int32)


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


def _basic_key(key, shape):
    """(y0, y1, x0, x1, keep_y, keep_x) of a zarr-style basic index on Y and X of ``shape``."""
    key = key if isinstance(key, tuple) else (key,)
    if len(key) > 3 or (len(key) == 3 and key[2] != slice(None)):
        raise IndexError('only Y and X can be indexed (the channel axis is read whole)')
    key = tuple(key) + (slice(None),) * (2 - min(len(key), 2))
    y0, y1, keep_y = _index(key[0], shape[0], 0)
    x0, x1, keep_x = _index(key[1], shape[1], 1)
    return y0, y1, x0, x1, keep_y, keep_x


def _getitem(arr, key):
    """``arr[key]`` as a host ndarray through ``arr.read_region`` (basic indexing on Y and X)."""
    y0, y1, x0, x1, keep_y, keep_x = _basic_key(key, arr.shape)
    out = np.empty((y1 - y0, x1 - x0, arr.shape[2]), dtype=np.uint8)
    if out.size:
        arr.read_region(y0, x0, y1 - y0, x1 - x0, out=out)
    return out[(slice(None) if keep_y else 0, slice(None) if keep_x else 0)]


def level_shape(shape, f):
    """Shape of the level-``f`` image of a Y x X x c array: ceil(Y/f) x ceil(X/f) x c."""
    return (-(-int(shape[0]) // f), -(-int(shape[1]) // f)) + tuple(int(s) for s in shape[2:])


def check_factor(f, ps):
    """``f`` as an int; ``ValueError`` unless it is a power of two with 1 <= f <= ps, ps % f == 0."""
    if isinstance(f, (bool, np.bool_)) or not isinstance(f, (int, np.integer)):
        raise ValueError('the downsample factor must be an int, got %r' % (f,))
    f = int(f)
    if f < 1 or f & (f - 1) or ps % f:
        raise ValueError('the downsample factor must be a power of two that divides the chunk '
                         'size %d, got %d' % (ps, f))
    return f


def reduce_plan(shape, ps, f, boxes, box_h, box_w):
    """``plan`` for boxes of the level-``f`` image of a Y x X x c array in ps^2 chunks.

    Every level pixel lies in one chunk (ps % f == 0), so the level image is stored in chunks of
    ps/f that correspond one to one with the level-0 chunks: ``chunk_yx`` names the same files.
    Returns ``(chunk_yx, pieces)`` with int32 P x 12 pieces ``{k, b, sy, sx, dy, dx, h, w, vh, vw,
    0, 0}``: ``plan``'s record in level pixels and the in-array extent of chunk k in level-0
    pixels, the record ``cae_tiles_crop_reduce_u8`` reads."""
    f = check_factor(f, ps)
    chunk_yx, p8 = plan(level_shape(shape, f), (ps // f, ps // f), boxes, box_h, box_w)
    iy, ix = chunk_yx[p8[:, 0], 0], chunk_yx[p8[:, 0], 1]
    pieces = np.zeros((len(p8), 12), dtype=np.int32)
    pieces[:, :8] = p8
    pieces[:, 8] = np.minimum(ps, int(shape[0]) - iy * ps)
    pieces[:, 9] = np.minimum(ps, int(shape[1]) - ix * ps)
    return chunk_yx, pieces


def check_levels(levels, ps):
    """``levels`` (K) as an int; ``ValueError`` unless K >= 1 and 2^K divides the chunk size."""
    if isinstance(levels, (bool, np.bool_)) or not isinstance(levels, (int, np.integer)):
        raise ValueError('levels must be an int, got %r' % (levels,))
    K = int(levels)
    if K < 1 or K > 30:
        raise ValueError('levels must be at least 1, got %d' % K)
    check_factor(2 ** K, ps)
    return K


def default_levels(shape, ps):
    """The smallest K >= 1 whose level image fits in one ps^2 chunk, capped at the largest K with
    2^K dividing ps (log2 ps for a power of two)."""
    cap = 0
    while ps % 2 ** (cap + 1) == 0:
        cap += 1
    K = 1
    while K < cap and max(level_shape(shape, 2 ** K)[:2]) > ps:
        K += 1
    return K


def pyramid_rows(gy, levels):
    """The level chunk rows in the order a pass over the gy level-0 chunk rows completes them:
    (k, R) once level-0 row 2^k (R + 1) - 1, or the last row, has been reduced."""
    return [(k, i >> k) for i in range(gy) for k in range(1, levels + 1)
            if (i + 1) % 2 ** k == 0 or i == gy - 1]


def pyramid_place(shape, ps, k, chunk_yx):
    """Where ``cae_tiles_pyramid_u8`` puts level-0 chunks ``chunk_yx`` (K x 2) of a Y x X array in
    ps^2 chunks at level k: int64 K x 5 ``{tile, oy, ox, eh, ew}``: tile column ``tile`` of level
    k's chunk row i >> k, at (oy, ox) in that tile, an in-array extent of eh x ew level pixels."""
    ij = np.asarray(chunk_yx, dtype=np.int64).reshape(-1, 2)
    i, j = ij[:, 0], ij[:, 1]
    f, lps = 2 ** k, ps >> k
    vh = np.minimum(ps, int(shape[0]) - i * ps)
    vw = np.minimum(ps, int(shape[1]) - j * ps)
    return np.stack([j >> k, (i % f) * lps, (j % f) * lps, -(-vh // f), -(-vw // f)], 1)


def pyramid_group(store, data_group):
    """The directory that holds the levels of the array ``<store>/<data_group>`` (``<group>`` of a
    ``<group>/0`` data group), or None when the data group's last component is not ``0``."""
    parts = [p for p in (data_group or '').split('/') if p]
    if not parts or parts[-1] != '0':
        return None
    return os.path.join(store, *parts[:-1])


class PyramidWriter:
    """Levels 1..K of a Y x X x c slide in ps^2 chunks whose level-0 tiles arrive in row-major
    order, batch by batch (``add``), each written as soon as it is complete.

    After each batch, ``cae_tiles_pyramid_u8`` reduces the batch's tiles into one chunk-row buffer
    per level (one launch per level-0 chunk row of the batch, so that rows of different level-1
    chunk rows never share the buffer).  Once the last level-0 row of a level chunk row has been
    reduced (``pyramid_rows`` order), its tiles are copied into a staging batch, which goes to
    ``encode(run)`` (a device uint8 run of ``batch`` tiles, fewer only at the end of a group -> its
    int32 symbols, in the current stream's order) whenever it is full: whole batches keep the
    encoder's buffers at one size.  The symbols are collected into coder groups
    (``_slide.group_sizes`` of the default schedule); each full group goes to
    ``code_and_write(sym, paths)`` with the chunk files ``level_path(k, (R, col, 0))`` of its
    tiles.  Beyond the caller's own memory this holds one chunk row per level, one batch of tiles
    and one group of symbols.  Everything runs on the current stream.  ``stage``: the device
    buffer of ``batch`` tiles to use as the staging batch (default a new one), so that a caller
    can replay a graph captured on it."""

    def __init__(self, shape, ps, levels, batch, device, level_path, encode, code_and_write,
                 sym_shape, stage=None):
        from ._slide import default_schedule, group_sizes
        self.shape, self.ps, self.levels, self.batch = tuple(shape), ps, levels, batch
        self.dev = device
        self.encode, self.code_and_write, self.sym_shape = encode, code_and_write, tuple(sym_shape)
        self.gy, self.gx = -(-int(shape[0]) // ps), -(-int(shape[1]) // ps)
        self.widths = [-(-self.gx // 2 ** k) for k in range(1, levels + 1)]
        self.first = np.concatenate([[0], np.cumsum(self.widths)]).astype(int)
        # one chunk row per level, back to back: the layout cae_tiles_pyramid_u8 writes
        self.rows = torch.zeros((int(self.first[-1]), ps, ps, int(shape[2])), dtype=torch.uint8,
                                device=device)
        self.order = pyramid_rows(self.gy, levels)
        self.paths = [level_path(k, (R, col, 0)) for k, R in self.order
                      for col in range(self.widths[k - 1])]
        self._groups = iter(group_sizes(len(self.paths), default_schedule(len(self.paths), batch),
                                        batch))
        self._gn, self._g0, self._lo, self._sym = next(self._groups), 0, 0, None
        self._x = stage if stage is not None else torch.empty(
            (batch, ps, ps, int(shape[2])), dtype=torch.uint8, device=device)
        self._fill = 0                  # tiles in the staging batch
        self._done = 0                  # level-0 chunk rows reduced so far
        self.flushed = []               # the level chunk rows handed to the encoder, in order
        self._recs_dev = torch.empty(4 * batch, dtype=torch.int32, device=device)

    def add(self, tiles, chunk_yx):
        """Reduce a batch: ``tiles`` (n x ps x ps x c uint8 on the device, contiguous) are the
        level-0 chunks ``chunk_yx`` (n x 2, row-major, after every chunk of earlier batches)."""
        ij = np.asarray(chunk_yx, dtype=np.int64).reshape(-1, 2)
        cuts = np.flatnonzero(np.diff(ij[:, 0])) + 1
        for a, b in zip(np.concatenate([[0], cuts]), np.concatenate([cuts, [len(ij)]])):
            self.complete(int(ij[a, 0]))         # the rows before this one are reduced
            self._launch(tiles, int(a), int(b), ij)

    def finish(self):
        """Write what is left once every level-0 chunk has been added."""
        self.complete(self.gy)

    def complete(self, upto):
        """Flush every level chunk row whose last level-0 row is below ``upto``."""
        for i in range(self._done, upto):
            for k in range(1, self.levels + 1):
                if (i + 1) % 2 ** k == 0 or i == self.gy - 1:
                    self._flush(k, i >> k)
        self._done = max(self._done, upto)

    def _launch(self, tiles, a, b, ij):
        ps, c = self.ps, int(self.shape[2])
        vh = np.minimum(ps, self.shape[0] - ij[a:b, 0] * ps)
        vw = np.minimum(ps, self.shape[1] - ij[a:b, 1] * ps)
        recs = np.ascontiguousarray(np.stack([ij[a:b, 0], ij[a:b, 1], vh, vw], 1), dtype=np.int32)
        C.check(C.lib().cae_tiles_pyramid_u8(
            tiles.data_ptr() + a * ps * ps * c, b - a, ps, c, self.levels, recs.ctypes.data,
            self._recs_dev.data_ptr(), self.gy, self.gx, self.rows.data_ptr(),
            _slide._stream_ptr(torch.cuda.current_stream(self.dev))))

    def _encode(self):
        n = self._fill
        if self._sym is None:
            self._sym = torch.empty((self._gn,) + self.sym_shape, dtype=torch.int32, device=self.dev)
        self._sym[self._g0:self._g0 + n].copy_(self.encode(self._x[:n]).reshape((n,) + self.sym_shape),
                                               non_blocking=True)
        self._g0 += n
        self._fill = 0
        if self._g0 == self._gn:
            self.code_and_write(self._sym, self.paths[self._lo:self._lo + self._gn])
            self._lo += self._gn
            self._gn, self._g0, self._sym = next(self._groups, 0), 0, None

    def _flush(self, k, R):
        """Encode level k's finished chunk row R, code every group it fills, clear the row."""
        row = self.rows[self.first[k - 1]:self.first[k]]
        a = 0
        while a < len(row):
            f = self._fill
            m = min(len(row) - a, self.batch - f, self._gn - self._g0 - f)
            self._x[f:f + m].copy_(row[a:a + m], non_blocking=True)
            self._fill += m
            a += m
            if self._fill == self.batch or self._g0 + self._fill == self._gn:
                self._encode()
        row.zero_()
        self.flushed.append((k, R))


def multiscales(levels, name=''):
    """The OME-Zarr 0.4 style ``multiscales`` entry of levels 0..K (axes y, x, c)."""
    return [{'version': '0.4', 'name': name,
             'axes': [{'name': 'y', 'type': 'space'}, {'name': 'x', 'type': 'space'},
                      {'name': 'c', 'type': 'channel'}],
             'datasets': [{'path': str(k), 'coordinateTransformations':
                           [{'type': 'scale', 'scale': [2 ** k, 2 ** k, 1]}]}
                          for k in range(levels + 1)],
             'type': 'mean'}]


def _write_json(path, obj):
    """``obj`` as JSON at ``path``, written aside and renamed: readers never see a partial file."""
    tmp = path + '.%d.tmp' % os.getpid()
    with open(tmp, 'w') as f:
        json.dump(obj, f, indent=1)
    os.replace(tmp, path)


def _read_attrs(group):
    try:
        with open(os.path.join(group, '.zattrs')) as f:
            return json.load(f)
    except FileNotFoundError:
        return {}


def stored_levels(group):
    """The level paths (ints) listed by the ``multiscales`` entry of ``<group>/.zattrs``; [0]
    without one."""
    ms = _read_attrs(group).get('multiscales')
    if not ms:
        return [0]
    return [int(d['path']) for d in ms[0]['datasets']]


def write_multiscales(store, group, levels):
    """``.zgroup`` at the store root and at ``group`` where absent, and the ``multiscales`` entry
    of levels 0..K in ``<group>/.zattrs`` (its other keys are kept; levels=0 removes the entry)."""
    for d in {os.path.normpath(store), os.path.normpath(group)}:
        if not os.path.exists(os.path.join(d, '.zgroup')):
            _write_json(os.path.join(d, '.zgroup'), {'zarr_format': 2})
    attrs = _read_attrs(group)
    attrs.pop('multiscales', None)
    if levels:
        attrs['multiscales'] = multiscales(levels)
    _write_json(os.path.join(group, '.zattrs'), attrs)


def _load_model(checkpoint, ps, c):
    """The model of ``checkpoint`` on the device, checked against chunks of ps x ps x c."""
    model = AE.autoencoder_from_state_dict(checkpoint, gpu=True, train=False)
    level = len(model['decoder'].module.synthesis_track)
    if ps % 2 ** level:
        raise ValueError('patch size %d is not a multiple of 2^%d' % (ps, level))
    last = model['decoder'].module.synthesis_track[-1]
    c_img = last.model[-1].out_channels if hasattr(last, 'model') else 3
    if c_img != c:
        raise ValueError('the model reconstructs %d channels, the array has %d' % (c_img, c))
    return model


def create_slide(path, checkpoint, shape, patch_size=512, data_group='0/0', overwrite=False,
                 **reader_kwargs):
    """Create an empty Y x X x C ``'cae'`` array and return a ``CompressedSlide`` open for
    writing (``mode='r+'``; ``reader_kwargs`` go to it).

    The ``.zarray`` is the one ``compress_image`` writes for the same arguments, and no chunk is
    written, so every chunk reads as the fill value 0 until it is assigned.  Assigning a slide
    strip by strip, in whole chunks, gives the files ``compress_image`` writes for the whole slide.
    An existing array is refused unless ``overwrite=True``, which removes its chunks as
    ``compress_image`` does."""
    from .compress import _CodecConfig, default_workers
    arr_path = os.path.join(path, data_group) if data_group else path
    if os.path.exists(os.path.join(arr_path, '.zarray')) and not overwrite:
        raise FileExistsError('%s already holds an array (pass overwrite=True to replace it)'
                              % arr_path)
    shape = tuple(int(s) for s in shape)
    ps = int(patch_size)
    if len(shape) != 3 or min(shape) <= 0 or ps <= 0:
        raise ValueError('expected a positive Y x X x C shape and patch size, got %r and %d'
                         % (shape, ps))
    _load_model(checkpoint, ps, shape[2])         # refuse a mismatched model before writing
    comp = _CodecConfig('cae', checkpoint=checkpoint if isinstance(checkpoint, str) else '<dict>',
                        gpu=False)
    arr = DirArray(arr_path, compressor=comp, mode='w', shape=shape, chunks=(ps, ps, shape[2]),
                   dtype=np.uint8)
    arr.remove_chunks(reader_kwargs.get('workers') or default_workers())
    return CompressedSlide(path, checkpoint, data_group=data_group, mode='r+', **reader_kwargs)


class CompressedSlide:
    """Random access to the pixels of a ``'cae'`` array written by ``compress_image``.

    ``path``: the store; ``data_group``: the array inside it; ``checkpoint``: the model it was
    compressed with (a path or a state dict); ``batch_tiles``: tiles per synthesis batch (the
    full batches replay a CUDA graph); ``workers``: native I/O and host coder threads;
    ``mode``: ``'r'`` (reads only) or ``'r+'`` (reads and writes: ``slide[...] = value``,
    ``write_region``, ``write_regions``).

    The reader owns its model and its device buffers, so it can run beside ``decompress_image``
    calls on other threads; calls on one reader are serialised, and a read after a write sees
    the new chunks.  Several processes may write to one array when their writes cover disjoint
    whole chunks; two that write a partly covered chunk at once may lose one of the writes (each
    reads, modifies and replaces the file, with no lock between processes).  The decode graphs
    (and with ``'r+'`` the encode graphs) are captured when the reader is opened."""

    def __init__(self, path, checkpoint, data_group='0/0', batch_tiles=16, workers=None, mode='r'):
        from .compress import default_workers
        if mode not in ('r', 'r+'):
            raise ValueError("mode must be 'r' or 'r+', got %r" % (mode,))
        if not torch.cuda.is_available():
            raise RuntimeError('CompressedSlide needs a CUDA device (no CPU fallback)')
        self._arr = DirArray(os.path.join(path, data_group) if data_group else path, mode='r')
        self._store = path
        self._data_group = data_group
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
        self.mode = mode
        model = _load_model(checkpoint, self.ps, self.shape[2])
        self.model = model
        self.fact_ent = model['fact_ent'].module
        self.workers = workers or default_workers()
        self.tc = _slide.TileCodec(model, self.ps, self.shape[2], int(batch_tiles),
                                   graphs=not os.environ.get('CAE_SLIDE_NO_GRAPHS'))
        self.tc.warm(encode=mode == 'r+', decode=True)
        self._tables = self.fact_ent._host_tables()
        self._pool = None
        self._pieces_dev = None
        self._uploaded = None             # the last upload out of the page-locked stream buffer
        self._lock = threading.Lock()
        self.stats = {}
        group = self._pyramid_group()
        self.levels = stored_levels(group) if group is not None else [0]

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
        return _getitem(self, key)

    def downsampled(self, f):
        """A read-only view of the slide at 1/``f`` of its resolution (``SlideLevel``): ``f`` is a
        power of two that divides the chunk size.  It shares this reader's model, buffers and
        lock, and reads see this reader's writes."""
        return SlideLevel(self, f)

    def level(self, k):
        """A read-only view of the stored pyramid level ``k`` (``<group>/k``, see
        ``build_pyramid``; ``StoredLevel``): the level's own chunks, read with this reader's
        model, buffers, lock and ``stats``.  ``level(0)`` is the slide itself.  Raises
        ``KeyError`` for a level that is not stored."""
        if isinstance(k, (bool, np.bool_)) or not isinstance(k, (int, np.integer)):
            raise TypeError('the level must be an int, got %r' % (k,))
        if int(k) not in self.levels:
            raise KeyError('level %d is not stored (stored levels: %s)' % (int(k), self.levels))
        return self if int(k) == 0 else StoredLevel(self, int(k))

    def _pyramid_group(self):
        """The directory holding the levels (``pyramid_group``), or None."""
        return pyramid_group(self._store, self._data_group)

    def build_pyramid(self, levels=None, overwrite=False):
        """Write the resolution pyramid: level k = 1..K as a ``'cae'`` array ``<group>/k`` beside
        the slide's ``<group>/0``, and a ``multiscales`` entry listing levels 0..K in
        ``<group>/.zattrs`` (``.zgroup`` files where absent).  Needs ``mode='r+'``.

        Level k holds ``self.downsampled(2 ** k)[:]`` (block means of the decoded slide, rounded
        half up; edge blocks average the pixels inside the array) encoded in ps^2 chunks with the
        slide's codec config: its ``.zarray`` and chunk files are the ones ``compress_image``
        writes for that image.  Reading a stored level (``level(k)``) decodes a few of its
        chunks instead of every level-0 chunk under the window, but its pixels went through one
        more lossy encode; ``downsampled(f)`` stays the exact mean of level 0.

        ``levels``: K, default the smallest K whose level fits in one chunk (capped at log2 ps).
        The slide is decoded once, group by group; after every synthesis batch one
        ``cae_tiles_pyramid_u8`` launch per level-0 chunk row in the batch reduces each decoded
        tile into every level, and each
        level chunk row is encoded, entropy-coded and written as soon as its last level-0 row has
        been reduced, so only one chunk row per level is ever held.  ``self.stats['decoded']``
        counts the level-0 chunk files read.

        The metadata follows OME-Zarr 0.4 ``multiscales`` (datasets with ``scale`` transforms
        [2^k, 2^k, 1], ``"type": "mean"``) with one difference: the axes are y, x, c, channel
        last as ``compress_image`` stores the slide, where OME-NGFF 0.4 puts the channel axis
        before the spatial ones.  The entry is written last, once every level file is; with
        ``overwrite=True`` the old entry is removed first, then the old levels' chunks, so a
        reader never finds a listed level with incomplete files.

        Later writes to the slide (``slide[...] = v``) do not update the levels: rebuild with
        ``overwrite=True`` after them.  Refused, before any file is touched: a reader opened with
        ``'r'``, K < 1 or 2^K not dividing ps, a data group whose last component is not ``0``,
        and existing level arrays unless ``overwrite=True``."""
        from .compress import _CodecConfig
        self._writable()
        ps, c = self.ps, self.shape[2]
        K = default_levels(self.shape, ps) if levels is None else check_levels(levels, ps)
        group = self._pyramid_group()
        if group is None:
            raise ValueError("the levels go beside a '<group>/0' array; this slide's data group "
                             "is %r" % (self._data_group,))
        level_paths = [os.path.join(group, str(k)) for k in range(1, K + 1)]
        existing = [q for q in level_paths if os.path.exists(os.path.join(q, '.zarray'))]
        if existing and not overwrite:
            raise FileExistsError('%s already holds a level array (pass overwrite=True to rebuild)'
                                  % existing[0])
        tc, B, dev = self.tc, self.tc.batch, self.tc.dev
        Y, X = self.shape[:2]
        gy, gx = self._arr.grid[:2]
        with self._lock, torch.cuda.device(dev):
            tc.warm(encode=False, decode=False, level=True)     # before the decode is in flight
            if overwrite:
                if 'multiscales' in _read_attrs(group):
                    write_multiscales(self._store, group, 0)
                    self.levels = [0]
                for q in existing:
                    DirArray(q, mode='r').remove_chunks(self.workers)
            cfg = dict(self._arr.compressor_config)
            comp = _CodecConfig(cfg.pop('id'), **cfg)
            arrs = {k: DirArray(q, compressor=comp, mode='w', shape=level_shape(self.shape, 2 ** k),
                                chunks=(ps, ps, c), dtype=np.uint8)
                    for k, q in zip(range(1, K + 1), level_paths)}
            for a in arrs.values():
                a.remove_chunks(self.workers)
            st = dict(device_coded=0)
            pyr = PyramidWriter(self.shape, ps, K, B, dev, lambda k, idx: arrs[k].chunk_file(idx),
                                lambda run: tc.encode_level(len(run)),
                                lambda sym, paths: self._code_and_write(sym, paths, st),
                                (tc.cb, tc.lh * tc.lw), stage=tc.level_stage())
            st['level_chunks'] = len(pyr.paths)

            def step(tiles, n_tiles, part):
                if tiles is None:        # missing chunks: their level pixels are the zeros rows holds
                    return
                pyr.add(tiles, part[:, 1:3])

            ii, jj = np.meshgrid(np.arange(gy), np.arange(gx), indexing='ij')
            chunk_yx = np.stack([ii.ravel(), jj.ravel()], 1)
            pieces = np.stack([np.arange(len(chunk_yx)), chunk_yx[:, 0], chunk_yx[:, 1],
                               np.minimum(ps, Y - chunk_yx[:, 0] * ps),
                               np.minimum(ps, X - chunk_yx[:, 1] * ps)], 1).astype(np.int32)
            self._decode_and_crop(chunk_yx, pieces, step)
            pyr.finish()
            torch.cuda.current_stream(dev).synchronize()
            self.stats.update(st)
            write_multiscales(self._store, group, K)
            self.levels = list(range(K + 1))

    # ---- public writes (mode='r+') ----
    def __setitem__(self, key, value):
        """zarr-style assignment on Y and X (the index as for ``__getitem__``).  ``value``: a
        Python int in [0, 255], a uint8 ndarray that broadcasts to the selection, or a contiguous
        uint8 CUDA tensor of the selection's shape.  Other dtypes are refused rather than cast.

        Like zarr, every chunk the selection touches is read, modified and re-encoded; a chunk
        the selection covers whole is encoded without reading it, and the re-encoding of a
        partly covered chunk is lossy (generation loss).  Unlike zarr, the padding of an edge
        chunk beyond the array edge is always stored as zeros, as ``compress_image`` stores it,
        so that writing a whole slide gives ``compress_image``'s files."""
        self._writable()
        y0, y1, x0, x1, keep_y, keep_x = _basic_key(key, self.shape)
        h, w, c = y1 - y0, x1 - x0, self.shape[2]
        sel = tuple(n for n, keep in ((h, keep_y), (w, keep_x)) if keep) + (c,)
        if isinstance(value, (bool, np.bool_)):
            raise TypeError('bool values are not uint8')
        if isinstance(value, (int, np.integer)):
            if not 0 <= int(value) <= 255:
                raise ValueError('%d does not fit in uint8' % int(value))
            if h and w:
                vals = torch.full((1, h, w, c), int(value), dtype=torch.uint8, device=self.tc.dev)
                self._write(np.array([[y0, x0]], dtype=np.int64), h, w, vals)
            return
        if isinstance(value, np.ndarray):
            if value.dtype != np.uint8:
                raise ValueError('values must be uint8, got %s (zarr would cast; this does not)'
                                 % value.dtype)
            try:
                value = np.broadcast_to(value, sel)
            except ValueError:
                raise ValueError('a value of shape %r does not broadcast to the selection %r'
                                 % (value.shape, sel)) from None
            if h and w:
                self._write(np.array([[y0, x0]], dtype=np.int64), h, w, value.reshape(1, h, w, c))
            return
        if isinstance(value, torch.Tensor):
            if h and w:
                self._write(np.array([[y0, x0]], dtype=np.int64), h, w,
                            self._device_values(value, sel).view(1, h, w, c))
            return
        raise TypeError('values must be an int, a uint8 ndarray or a uint8 CUDA tensor, got %s'
                        % type(value).__name__)

    def write_regions(self, boxes, h, w, values):
        """Write the ``h`` x ``w`` windows with top-left corners ``boxes`` ((y, x) pairs):
        ``values`` is an N x h x w x c uint8 CUDA tensor or host ndarray (page-locked ones are
        uploaded asynchronously).  Overlapping boxes are refused before any file is touched.
        Chunks are re-encoded as for ``__setitem__``."""
        self._writable()
        yx = np.asarray(boxes, dtype=np.int64).reshape(-1, 2)
        shape = (len(yx), int(h), int(w), self.shape[2])
        if isinstance(values, torch.Tensor):
            values = self._device_values(values, shape)
        elif isinstance(values, np.ndarray):
            if values.dtype != np.uint8 or values.shape != shape:
                raise ValueError('values must be a uint8 ndarray of shape %r, got %s %r'
                                 % (shape, values.dtype, values.shape))
        else:
            raise TypeError('values must be a uint8 CUDA tensor or host ndarray')
        self._write(yx, int(h), int(w), values)

    def write_region(self, y, x, value):
        """Write one h x w x c window at (y, x); ``value`` as one window of ``write_regions``."""
        self._writable()
        if not isinstance(value, (torch.Tensor, np.ndarray)) or value.ndim != 3:
            raise ValueError('value must be an h x w x c uint8 CUDA tensor or host ndarray')
        self.write_regions([(y, x)], value.shape[0], value.shape[1], value[None])

    def _writable(self):
        if self.mode != 'r+':
            raise ValueError("this slide was opened for reading; open it with mode='r+' to write")

    def _device_values(self, t, shape):
        if (tuple(t.shape) != tuple(shape) or t.dtype != torch.uint8 or t.device != self.tc.dev
                or not t.is_contiguous()):
            raise ValueError('values must be a contiguous uint8 tensor of shape %r on %s, got %s '
                             '%r on %s' % (tuple(shape), self.tc.dev, t.dtype, tuple(t.shape),
                                           t.device))
        return t

    def close(self):
        if self._pool is not None:
            self._pool.shutdown()
            self._pool = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- the work ----
    def _read(self, yx, h, w, out, shape, f=1, arr=None):
        """The boxes ``yx`` of the level-``f`` image (f = 1: the slide, or the stored array
        ``arr``) into ``out``."""
        n_boxes = len(yx)
        arr = self._arr if arr is None else arr
        if f == 1:
            chunk_yx, pieces = plan(arr.shape, arr.chunks, yx, h, w)
        else:
            chunk_yx, pieces = reduce_plan(self.shape, self.ps, f, yx, h, w)
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
        if f == 1:
            def step(tiles, n_tiles, part):
                self._crop(tiles, n_tiles, part, dst, n_boxes, h, w)
        else:
            def step(tiles, n_tiles, part):
                self._crop_reduce(tiles, n_tiles, f, part, dst, n_boxes, h, w)
        with self._lock, torch.cuda.device(dev):
            self._decode_and_crop(chunk_yx, pieces, step, arr)
            if host_out is None:
                return dst
            if _slide.is_pinned_array(host_out):
                torch.from_numpy(host_out).copy_(dst, non_blocking=True)
                torch.cuda.current_stream(dev).synchronize()
            else:
                torch.from_numpy(host_out).copy_(dst)
            return host_out

    def _table(self, pieces):
        """The piece table as a contiguous int32 host array, and a device buffer large enough for
        it (the table goes up on the launch's stream, so one device buffer serves every launch)."""
        if self._pieces_dev is None or self._pieces_dev.numel() < pieces.size:
            self._pieces_dev = torch.empty(max(8 * 1024, pieces.size), dtype=torch.int32,
                                           device=self.tc.dev)
        return np.ascontiguousarray(pieces, dtype=np.int32)

    def _crop(self, tiles, n_tiles, pieces, dst, n_boxes, h, w):
        """One ``cae_tiles_crop_u8`` launch on the current stream."""
        pieces = self._table(pieces)
        C.check(C.lib().cae_tiles_crop_u8(
            tiles.data_ptr() if tiles is not None else None, n_tiles, self.ps, self.tc.c_img,
            pieces.ctypes.data, len(pieces), self._pieces_dev.data_ptr(), dst.data_ptr(),
            n_boxes, h, w, _slide._stream_ptr(torch.cuda.current_stream(self.tc.dev))))

    def _crop_reduce(self, tiles, n_tiles, f, pieces, dst, n_boxes, h, w):
        """One ``cae_tiles_crop_reduce_u8`` launch on the current stream (``pieces``: P x 12)."""
        pieces = self._table(pieces)
        C.check(C.lib().cae_tiles_crop_reduce_u8(
            tiles.data_ptr() if tiles is not None else None, n_tiles, self.ps, self.tc.c_img, f,
            pieces.ctypes.data, len(pieces), self._pieces_dev.data_ptr(), dst.data_ptr(),
            n_boxes, h, w, _slide._stream_ptr(torch.cuda.current_stream(self.tc.dev))))

    def _paste(self, tiles, n_tiles, pieces, values, h, w):
        """One ``cae_tiles_paste_u8`` launch on the current stream."""
        pieces = self._table(pieces)
        C.check(C.lib().cae_tiles_paste_u8(
            tiles.data_ptr(), n_tiles, self.ps, self.tc.c_img, pieces.ctypes.data, len(pieces),
            self._pieces_dev.data_ptr(), values.data_ptr(), values.shape[0], h, w,
            _slide._stream_ptr(torch.cuda.current_stream(self.tc.dev))))

    def _present(self, chunk_yx, arr=None):
        """Chunk file paths of ``chunk_yx`` (of ``arr``, default the slide) and which of them
        exist."""
        paths = [(self._arr if arr is None else arr).chunk_file((int(i), int(j), 0)) for i, j in chunk_yx]
        sizes = np.empty(len(paths), dtype=np.int64)
        C.check(C.lib().cae_files_stat(_paths_blob(paths), len(paths), sizes.ctypes.data,
                                       self.workers))
        return paths, sizes >= 0

    def _decode_streams(self, paths, st):
        """Read the chunk files ``paths`` (one coder group) and entropy-decode their streams:
        the device coder from ``GPU_CODER_MIN_STREAMS`` streams up, host coder threads below.
        Returns the int32 symbols n x cb x lh x lw on the device (ready in the current stream's
        order) and the device coder's status tensor (None for the host coder), which the caller
        checks once it has synchronised.  Raises before any decode if a header is not the
        (patch, patch) the codec writes."""
        tc, fe, dev, gn = self.tc, self.fact_ent, self.tc.dev, len(paths)
        if self._uploaded is not None:
            self._uploaded.synchronize()      # the page-locked buffer's last upload has left it
        hdr, payload, off = native_read(paths, 16, self.workers,
                                        alloc=lambda n: tc.pinned('region_streams', n).numpy())
        if bytes(hdr[0]) != struct.pack('>QQ', self.ps, self.ps) or (hdr != hdr[0]).any():
            raise C.CaeError('chunk headers differ from the (patch, patch) the codec wrote')
        status = None
        if gn >= fe.GPU_CODER_MIN_STREAMS:
            if (off % 4).any():
                raise C.CaeError('chunk streams are not whole words')
            words = torch.empty(int(off[-1]) // 4, dtype=torch.int32, device=dev)
            words.view(torch.uint8).copy_(torch.from_numpy(payload), non_blocking=True)
            sym, status = fe.decode_streams_device(words, off // 4, tc.lh * tc.lw,
                                                   defer_status=True)
            st['device_decoded'] += gn
        else:
            # few streams: one host thread per stream beats the device coder's fixed cost
            cdf, sz, offs = self._tables
            sym = np.stack(list(self._threads().map(
                lambda k: decode_symbols(payload[off[k]:off[k + 1]], tc.cb, tc.lh * tc.lw,
                                         cdf, sz, offs), range(gn))))
            sym = torch.from_numpy(sym).pin_memory().to(dev, non_blocking=True)
        self._uploaded = torch.cuda.Event()
        self._uploaded.record(torch.cuda.current_stream(dev))
        st['decoded'] += gn
        return sym.reshape(gn, tc.cb, tc.lh, tc.lw), status

    def _threads(self):
        if self._pool is None:
            self._pool = ThreadPoolExecutor(max_workers=self.workers)
        return self._pool

    def _decode_and_crop(self, chunk_yx, pieces, step, arr=None):
        """Decode the chunks ``chunk_yx`` (of ``arr``, default the slide) group by group (``_slide.group_sizes``: the symbols of
        at most one group are on the device) and hand every synthesis batch with its ``pieces``
        to ``step(tiles, n_tiles, part)`` on the current stream (``part[:, 0]`` indexes the
        batch; the pieces of missing chunks come first, with ``tiles`` None and k = -1).
        Returns once the device is done."""
        tc, fe = self.tc, self.fact_ent
        B, dev = tc.batch, tc.dev
        main = torch.cuda.current_stream(dev)
        paths, present = self._present(chunk_yx, arr)   # a missing chunk reads as the fill value 0
        # position of every chunk among the decoded ones (-1: missing), per piece
        piece_tile = np.where(present, np.cumsum(present) - 1, -1)[pieces[:, 0]]
        if not present.all():
            fill = pieces[piece_tile < 0].copy()
            fill[:, 0] = -1
            step(None, 0, fill)
        todo = [paths[k] for k in np.nonzero(present)[0]]
        self.stats = st = dict(chunks=len(paths), decoded=0, device_decoded=0,
                               missing=len(paths) - len(todo))
        statuses = []
        slot = lo = 0
        groups = _slide.group_sizes(len(todo), _slide.default_schedule(len(todo), B, decode=True),
                                    B) if todo else []
        for gn in groups:
            sym, status = self._decode_streams(todo[lo:lo + gn], st)
            if status is not None:
                statuses.append(status)
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
                step(u8, n, part)
            lo += gn
        main.synchronize()
        for status in statuses:
            fe.check_decode_status(status)

    def _write(self, yx, h, w, values):
        """Write the boxes ``yx`` (``values``: N x h x w x c, on the device or the host) chunk by
        chunk: group by group (``_slide.group_sizes``), the group's partly covered chunks that
        have a file are read and decoded, every synthesis-sized batch is assembled in a slot of
        the codec (decoded tiles, zeros for missing partly covered chunks, then one
        ``cae_tiles_paste_u8`` launch for the new pixels and the zero padding), encoded, and
        the group's streams are entropy-coded and written as chunk files (.partial, renamed).
        Nothing is written before the boxes and values are checked, and a group's files are
        only written once its old chunks have decoded cleanly."""
        chunk_yx, pieces, full, fill = write_plan(self.shape, self.chunks, yx, h, w)
        tc, fe = self.tc, self.fact_ent
        B, dev = tc.batch, tc.dev
        with self._lock, torch.cuda.device(dev):
            main = torch.cuda.current_stream(dev)
            if isinstance(values, torch.Tensor):
                vals = values
            elif _slide.is_pinned_array(values):
                vals = torch.from_numpy(values).to(dev, non_blocking=True)
            else:
                vals = torch.from_numpy(np.ascontiguousarray(values)).to(dev)
            paths, present = self._present(chunk_yx)
            # work order: partly covered chunks with a file (decoded), partly covered missing
            # ones (zeroed), fully covered ones (pasted over whatever the slot held); in every
            # batch the decoded tiles are then a prefix, moved in with one device copy
            kind = np.where(full, 2, np.where(present, 0, 1))
            order = np.argsort(kind, kind='stable')
            kind = kind[order]
            pos = np.empty_like(order)
            pos[order] = np.arange(len(order))
            table = np.concatenate([pieces, fill])
            table_pos = pos[table[:, 0]]
            srt = np.argsort(table_pos, kind='stable')
            table, table_pos = table[srt], table_pos[srt]
            K = len(chunk_yx)
            self.stats = st = dict(chunks=K, full=int(full.sum()), partial=int(K - full.sum()),
                                   decoded=0, device_decoded=0, missing=int(K - present.sum()),
                                   device_coded=0)
            slot = lo = 0
            for gn in _slide.group_sizes(K, _slide.default_schedule(K, B), B):
                gd = int((kind[lo:lo + gn] == 0).sum())
                gz = int((kind[lo:lo + gn] == 1).sum())
                old, status = (self._decode_streams([paths[k] for k in order[lo:lo + gd]], st)
                               if gd else (None, None))
                sym_out = torch.empty((gn, tc.cb, tc.lh * tc.lw), dtype=torch.int32, device=dev)
                for p0 in range(0, gn, B):
                    n = min(B, gn - p0)
                    x = tc.x[slot]
                    nd = min(max(gd - p0, 0), n)
                    if nd == B and tc.graphs:
                        tc.sym_in[slot].copy_(old[p0:p0 + nd], non_blocking=True)
                        x.copy_(tc.decode(slot, nd), non_blocking=True)
                    elif nd:
                        x[:nd].copy_(tc.decode_eager(old[p0:p0 + nd]), non_blocking=True)
                    nz = min(max(gd + gz - p0, 0), n) - nd
                    if nz:
                        x[nd:nd + nz].zero_()
                    a, b = np.searchsorted(table_pos, [lo + p0, lo + p0 + n])
                    part = table[a:b].copy()
                    part[:, 0] = table_pos[a:b] - (lo + p0)
                    self._paste(x, n, part, vals, h, w)
                    sym_out[p0:p0 + n].copy_(tc.encode(slot, n).reshape(n, tc.cb, -1),
                                             non_blocking=True)
                    slot = (slot + 1) % tc.slots
                self._code_and_write(sym_out, [paths[k] for k in order[lo:lo + gn]], st, status)
                lo += gn
            main.synchronize()


    def _code_and_write(self, sym_out, paths, st, status=None):
        """Entropy-code the symbols ``sym_out`` (n x cb x lh*lw on the device, complete in the
        current stream's order) of one group and write them as the chunk files ``paths``
        (.partial, renamed): the device coder from ``GPU_CODER_MIN_STREAMS`` streams up, host
        coder threads below.  ``status``: the device decoder's status of the group's old chunks,
        checked before any file is written."""
        _, device_coded = _slide.code_and_write(
            self.fact_ent, self._tables, sym_out, paths, self.ps, self.workers,
            lambda n: self.tc.pinned('region_write_streams', n), self._threads(), status)
        st['device_coded'] += device_coded

class SlideLevel:
    """The slide at 1/``f`` of its resolution (``CompressedSlide.downsampled(f)``), read-only.

    The level-``f`` image of a Y x X x c slide is ceil(Y/f) x ceil(X/f) x c.  Its pixel (i, j),
    channel ch, is the mean, rounded half up, of the slide's pixels in rows [i f, min((i+1) f, Y))
    x columns [j f, min((j+1) f, X)): what PIL's ``Image.reduce(f)`` computes on whole blocks,
    while edge blocks average only the pixels inside the array.  A missing chunk reads as 0.

    Reads decode the chunks they touch exactly as the slide's own reads do (same files, coder
    groups, synthesis batches, lock and ``stats``); after every synthesis batch one
    ``cae_tiles_crop_reduce_u8`` launch writes the batch's pieces of the level image, so no
    buffer of the level-0 window exists.  ``f`` = 1 reads the slide through its own path."""

    def __init__(self, slide, f):
        self.downsample = check_factor(f, slide.ps)
        self._slide = slide
        self.shape = level_shape(slide.shape, self.downsample)
        self.chunks = (slide.ps // self.downsample,) * 2 + (slide.shape[2],)
        self.dtype = slide.dtype

    def read_regions(self, boxes, h, w, out=None):
        """The ``h`` x ``w`` windows at ``boxes`` of the level image; as the slide's
        ``read_regions``, in level pixels."""
        yx = np.asarray(boxes, dtype=np.int64).reshape(-1, 2)
        return self._slide._read(yx, int(h), int(w), out, (len(yx), int(h), int(w), self.shape[2]),
                                 self.downsample)

    def read_region(self, y, x, h, w, out=None):
        """One ``h`` x ``w`` x c window at (y, x) of the level image; ``out`` as for
        ``read_regions``."""
        return self._slide._read(np.array([[y, x]], dtype=np.int64), int(h), int(w), out,
                                 (int(h), int(w), self.shape[2]), self.downsample)

    def __getitem__(self, key):
        """zarr-style basic indexing on Y and X of the level image: a host ndarray."""
        return _getitem(self, key)

    def __setitem__(self, key, value):
        raise TypeError('a downsampled view is read-only: write to the slide it was taken from')


class StoredLevel:
    """A stored pyramid level (``CompressedSlide.level(k)``), read-only: the ``'cae'`` array
    ``<group>/k`` that ``build_pyramid`` wrote, read with the slide's model, buffers, lock, pool
    and ``stats`` (switching levels captures no graphs and loads no model).  Its pixels are the
    ones a ``CompressedSlide`` opened on ``data_group='<group>/k'`` reads."""

    def __init__(self, slide, k):
        self._slide = slide
        self._arr = DirArray(os.path.join(slide._pyramid_group(), str(k)), mode='r')
        self.downsample = 2 ** k
        self.shape, self.chunks, self.dtype = self._arr.shape, self._arr.chunks, self._arr.dtype
        want = level_shape(slide.shape, self.downsample)
        if ((self._arr.compressor_config or {}).get('id') != 'cae' or self.shape != want
                or self.chunks != slide.chunks or self.dtype != slide.dtype):
            raise ValueError('%s is not a level %d of this slide: expected a %r uint8 \'cae\' '
                             'array in %r chunks' % (self._arr.path, k, want, slide.chunks))

    def read_regions(self, boxes, h, w, out=None):
        """The ``h`` x ``w`` windows at ``boxes`` of the level; as the slide's ``read_regions``,
        in level pixels."""
        yx = np.asarray(boxes, dtype=np.int64).reshape(-1, 2)
        return self._slide._read(yx, int(h), int(w), out, (len(yx), int(h), int(w), self.shape[2]),
                                 arr=self._arr)

    def read_region(self, y, x, h, w, out=None):
        """One ``h`` x ``w`` x c window at (y, x) of the level; ``out`` as for
        ``read_regions``."""
        return self._slide._read(np.array([[y, x]], dtype=np.int64), int(h), int(w), out,
                                 (int(h), int(w), self.shape[2]), arr=self._arr)

    def __getitem__(self, key):
        """zarr-style basic indexing on Y and X of the level: a host ndarray."""
        return _getitem(self, key)

    def __setitem__(self, key, value):
        raise TypeError('a stored level is read-only: write to the slide and rebuild the pyramid')
