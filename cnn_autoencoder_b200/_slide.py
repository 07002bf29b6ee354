"""Batched whole-slide engine behind ``compress_image`` / ``decompress_image``.

The reference walks a slide one ``patch_size`` chunk at a time: dask hands each chunk to the
codec (``src/compress.py:101-128``, ``src/models/tasks/_autoencoders.py:539-555``), whose
``encode`` runs the analysis transform at batch 1, copies the latent to the host, turns it into
a Python list and entropy-codes it on one thread; ``decompress.py:72-96`` mirrors that.  This
module does the same work B200-first:

* tiles move between the row-major slide in page-locked host memory and tile-major device
  buffers as strided DMA copies (``cae_tiles_upload_u8`` / ``cae_tiles_download_u8``): no
  host-side gather, no staging copy; three buffer slots keep upload, kernels and download of
  neighbouring batches in flight on three CUDA streams;
* one *batch* of tiles runs the analysis transform + quantizer (or de-quantizer + synthesis
  transform) as one CUDA-graph replay;
* the integer symbols of a whole *group* of tiles (up to ``coder_tiles``) stay on the device
  and all their rANS streams are coded at once (a stream is sequential: the parallelism is
  across tiles) on a second stream while the transforms of the next group run;
* only the packed streams (~0.6 byte per pixel) cross PCIe in the compressed direction, and
  native threads write / read the chunk files.

Everything here is plumbing around kernels of ``libcae_b200.so``; there is no CPU fallback.
"""
import contextlib
import ctypes
import struct
import threading
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

from . import _cabi as C
from . import _ops as O
from ._entropy import encode_symbols
from ._store import native_gather, native_read, native_write


def is_pinned_array(arr):
    """True for a C-contiguous uint8 ndarray living in page-locked memory (a ``torch`` pinned
    tensor's ``.numpy()`` view, or memory registered with ``pin_array``)."""
    if not (isinstance(arr, np.ndarray) and arr.dtype == np.uint8 and arr.flags.c_contiguous):
        return False
    if arr.size == 0 or not torch.cuda.is_available():
        return False
    try:
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')          # read-only arrays: we only ask where they live
            return bool(torch.from_numpy(arr.reshape(-1)[:1]).is_pinned())
    except (RuntimeError, ValueError, TypeError):
        return False


def _tiles_pinned(src, tile_yx, ps):
    """Are the rows of ``src`` that the tiles touch page-locked?  (A rank may have locked only
    the rows of its own shard of a slide.)"""
    if not (isinstance(src, np.ndarray) and src.dtype == np.uint8 and src.flags.c_contiguous
            and src.ndim == 3 and len(tile_yx)):
        return False
    y_lo = int(tile_yx[:, 0].min()) * ps
    y_hi = min(src.shape[0], (int(tile_yx[:, 0].max()) + 1) * ps)
    return is_pinned_array(src[y_lo:y_lo + 1]) and is_pinned_array(src[y_hi - 1:y_hi])


def pin_array(arr):
    """Page-lock an existing ndarray in place (``cudaHostRegister``) so tiles can be DMA'd
    straight out of / into it.  Returns a handle whose ``close()`` unregisters."""
    rt = torch.cuda.cudart()
    err = rt.cudaHostRegister(arr.ctypes.data, arr.nbytes, 0)
    if int(err) != 0:
        raise C.CaeError('cudaHostRegister failed (%s)' % err)

    class _Handle:
        def close(self_inner):
            rt.cudaHostUnregister(arr.ctypes.data)
    return _Handle()


def _stream_ptr(s):
    return ctypes.c_void_p(s.cuda_stream)


@torch.no_grad()
def encode_tiles(enc, fe, x):
    """The analysis transform ``enc`` and the quantizer of the entropy bottleneck ``fe`` on uint8
    tiles N x ps x ps x c (device, current stream) -> int32 symbols N x C x lh x lw."""
    _, _, sym, _, _ = fe._quantize_cuda(enc(x), want_yq=False, want_p=False, want_sym=True)
    return sym


class TileCodec:
    """The device side for one model and one tile size: ``slots`` input / output buffer slots of
    ``batch`` tiles each, the per-batch kernels captured in CUDA graphs (one per slot)."""

    def __init__(self, model, ps, c_img, batch, slots=3, graphs=True):
        self.enc, self.dec = model['encoder'], model['decoder']
        self.fe = model['fact_ent'].module
        self.dev = next(self.enc.parameters()).device
        self.ps, self.c_img, self.batch, self.slots = ps, c_img, batch, slots
        self.level = len(self.dec.module.synthesis_track)
        if ps % (2 ** self.level):
            raise C.CaeError('patch size %d is not a multiple of 2^%d' % (ps, self.level))
        self.lh = self.lw = ps // 2 ** self.level
        self.cb = self.fe.channels
        self.graphs = graphs
        self.x = [torch.empty((batch, ps, ps, c_img), dtype=torch.uint8, device=self.dev)
                  for _ in range(slots)]
        self.sym_in = [torch.empty((batch, self.cb, self.lh, self.lw), dtype=torch.int32,
                                   device=self.dev) for _ in range(slots)]
        self._enc_g = [None] * slots      # (graph, static symbols out)
        self.x_level = None               # staging batch of pyramid level tiles (encode_level)
        self._lvl_g = None                # (graph, static symbols out) of x_level
        self._dec_g = [None] * slots      # (graph, static uint8 out)
        self._keep = []
        self.launches_enc = self.launches_dec = 0
        self.replays_enc = self.replays_dec = 0
        self._pins = {}              # page-locked staging buffers, kept across calls
        # streams live as long as the codec: the caching allocator pools memory per stream, so a
        # fresh stream per call would cudaMalloc its gigabyte-sized scratch again every time
        self.s_in, self.s_out, self.s_code = (torch.cuda.Stream(self.dev) for _ in range(3))
        # the decoder's own coder stream: a decompress_image call may run beside a compress_image
        # call on the same model (two slides in flight, each call on its own thread and stream)
        self.s_dec = torch.cuda.Stream(self.dev)
        self._bufs = {}

    # ---- the per-batch work, eager form (also what the graphs capture) ----
    def encode_eager(self, x):
        """uint8 N x ps x ps x c (device) -> int32 symbols N x C x lh x lw."""
        return encode_tiles(self.enc, self.fe, x)

    @torch.no_grad()
    def decode_eager(self, sym):
        """int32 symbols N x C x lh x lw (device) -> uint8 N x ps x ps x c."""
        n = sym.shape[0]
        key = (n, str(self.dev))
        buf = getattr(self, '_planar', {}).get(key)
        if buf is None:
            buf = O.alloc_act(C.FMT_F16_PLANAR, n, self.cb, self.lh, self.lw, C.HALO_KEEP,
                              device=self.dev)
            self.__dict__.setdefault('_planar', {})[key] = buf
        med = self.fe._device_tables()['medians']
        C.check(C.lib().cae_eb_dequantize_planar(sym.data_ptr(), med.data_ptr(), n, self.cb,
                                                 self.lh, self.lw, buf.desc(),
                                                 _stream_ptr(torch.cuda.current_stream(self.dev))))
        _, _, u8 = self.dec.module.forward_planar(buf, as_uint8='only')
        return u8

    def _capture(self, fn, arg):
        side = torch.cuda.Stream(self.dev)
        side.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(side):
            for _ in range(2):
                fn(arg)
        torch.cuda.current_stream(self.dev).wait_stream(side)
        torch.cuda.synchronize(self.dev)
        g = torch.cuda.CUDAGraph()
        n0 = C.launch_count()
        with torch.cuda.graph(g):
            out = fn(arg)
        launches = C.launch_count() - n0
        # the graph holds raw pointers into the executors' cached buffers
        self._keep.append([dict(m.module._executor()._buffers) for m in (self.enc, self.dec)])
        return g, out, launches

    def encode(self, slot, n):
        """Run the analysis transform + quantizer on ``self.x[slot][:n]`` (current stream);
        returns the symbols (valid until the slot is encoded again)."""
        if n == self.batch and self.graphs:
            if self._enc_g[slot] is None:
                g, out, self.launches_enc = self._capture(self.encode_eager, self.x[slot])
                self._enc_g[slot] = (g, out)
            g, out = self._enc_g[slot]
            g.replay()
            self.replays_enc += 1
            return out
        return self.encode_eager(self.x[slot][:n])

    def encode_level(self, n):
        """``encode`` of ``self.level_stage()[:n]``, the staging batch of ``region.PyramidWriter``
        (its own graph: the upload slots belong to the tile loop's upload stream)."""
        if n == self.batch and self.graphs:
            if self._lvl_g is None:
                g, out, _ = self._capture(self.encode_eager, self.level_stage())
                self._lvl_g = (g, out)
            g, out = self._lvl_g
            g.replay()
            return out
        return self.encode_eager(self.level_stage()[:n])

    def level_stage(self):
        if self.x_level is None:
            self.x_level = torch.empty((self.batch, self.ps, self.ps, self.c_img),
                                       dtype=torch.uint8, device=self.dev)
        return self.x_level

    def decode(self, slot, n):
        """Run de-quantizer + synthesis transform on ``self.sym_in[slot][:n]``; returns the uint8
        tiles (valid until the slot is decoded again)."""
        if n == self.batch and self.graphs:
            if self._dec_g[slot] is None:
                g, out, self.launches_dec = self._capture(self.decode_eager, self.sym_in[slot])
                self._dec_g[slot] = (g, out)
            g, out = self._dec_g[slot]
            g.replay()
            self.replays_dec += 1
            return out
        return self.decode_eager(self.sym_in[slot][:n])

    def buffer(self, name, shape, dtype):
        """A device tensor kept under ``name`` (reallocated when the shape changes)."""
        t = self._bufs.get(name)
        if t is None or tuple(t.shape) != tuple(shape) or t.dtype != dtype:
            t = self._bufs[name] = torch.empty(shape, dtype=dtype, device=self.dev)
        return t

    def pinned(self, name, nbytes):
        """A page-locked uint8 buffer of at least ``nbytes`` kept under ``name`` (page-locking
        is slow and stalls other CUDA calls: allocate once, grow rarely)."""
        buf = self._pins.get(name)
        if buf is None or buf.numel() < nbytes:
            buf = self._pins[name] = torch.empty(int(nbytes * 1.3) + 4096, dtype=torch.uint8,
                                                 pin_memory=True)
        return buf[:nbytes]

    def warm(self, encode=True, decode=True, level=False):
        """Build the graphs of every slot (and with ``level`` the one of ``encode_level``) up
        front (outside any timed region)."""
        if not self.graphs:
            return
        built = False
        if level and self._lvl_g is None:
            self.encode_level(self.batch)
            built = True
        for s in range(self.slots):
            if encode and self._enc_g[s] is None:
                self.encode(s, self.batch)
                built = True
            if decode and self._dec_g[s] is None:
                self.decode(s, self.batch)
                built = True
        if built:
            torch.cuda.synchronize(self.dev)


_codecs = {}
_codecs_lock = threading.Lock()


def tile_codec(model, ps, c_img, batch, graphs=None):
    """One TileCodec per (model dict, tile size, batch): graphs and buffers are reused across
    calls of the tile loops on the same model."""
    if graphs is None:
        import os
        graphs = not os.environ.get('CAE_SLIDE_NO_GRAPHS')
    key = (id(model['encoder']), id(model['decoder']), id(model['fact_ent']), ps, c_img, batch,
           graphs)
    with _codecs_lock:
        tc = _codecs.get(key)
        if tc is None:
            if len(_codecs) > 4:
                _codecs.clear()
            tc = _codecs[key] = TileCodec(model, ps, c_img, batch, graphs=graphs)
            tc._model = model            # keeps the ids above valid
        return tc


class _Stats(dict):
    def add(self, k, v):
        self[k] = self.get(k, 0) + v


def group_sizes(n_tiles, coder_tiles, batch):
    """How the tiles of a shard are split into entropy-coder groups.  ``coder_tiles`` is either
    one size (equal groups) or a sequence of sizes, the last of which repeats: a coder call
    costs the same whatever its stream count, so few groups are best for the device, but what
    follows the LAST group of ``compress_tiles`` (its coder call, the stream download and its
    chunk-file writes) and what precedes the FIRST group of ``decompress_tiles`` (file reads,
    upload, decode) has nothing to hide under -- an uneven schedule such as (6144, 2048) keeps
    the exposed group of ``compress_tiles`` small.  Every size is rounded up to whole batches."""
    seq = [coder_tiles] if isinstance(coder_tiles, (int, np.integer)) else list(coder_tiles)
    if not seq or any(int(g) <= 0 for g in seq):
        raise ValueError('coder_tiles must be a positive size or a non-empty sequence of them')
    sizes, left, k = [], n_tiles, 0
    while left > 0:
        g = int(seq[min(k, len(seq) - 1)])
        g = -(-max(batch, g) // batch) * batch
        g = min(g, left)
        sizes.append(g)
        left -= g
        k += 1
    return sizes


def default_schedule(n_tiles, batch, decode=False, cap=8192):
    """The group schedule the tile loops use when the caller names none (``coder_tiles=None``).
    Measured on a B200 at 8192 chunks of 512^2 (``tools/micro/trace_slide.py``, DESIGN 6.9): a
    coder call costs 19 ms (encode) / 33 ms (decode) whatever its size and its blocks keep the
    transforms' persistent kernels off their SMs meanwhile, so groups are few and large (at most
    ``cap`` tiles: 6.4 GB of symbols).  What follows the last group of ``compress_tiles`` (coder
    call, stream download, chunk-file writes) has nothing to hide under, so from 6144 tiles on the
    shard is split 3 : 1 -- (6144, 2048): 318 ms, (4096, 4096): 350 ms, one group: 351 ms, (4096,
    3072, 1024): 324-336 ms; for ``decompress_tiles`` two equal groups measured best (200-211 ms
    against 220-239 ms for five tapered alternatives).  Shards under 2048 tiles are one group."""
    if n_tiles < 2048:
        return [max(batch, n_tiles)]
    if decode or n_tiles < 6144:
        n_groups = max(2, -(-n_tiles // cap))
        return group_sizes(n_tiles, -(-n_tiles // n_groups), batch)
    sizes, left = [], n_tiles
    while left > cap * 4 // 3:
        sizes.append(cap)
        left -= cap
    tail = max(batch, left // 4 // batch * batch)
    return group_sizes(n_tiles, sizes + [left - tail, tail], batch)


def code_and_write(fe, tables, sym, paths, ps, workers, pinned, pool, status=None,
                   lock=contextlib.nullcontext()):
    """Entropy-code the symbols ``sym`` (n x cb x lh*lw on the device, complete in the current
    stream's order) of one group and write them as the ps^2 chunk files ``paths`` (.partial,
    renamed): the device coder from ``fe.GPU_CODER_MIN_STREAMS`` streams up (its packed streams
    come back through the page-locked buffer ``pinned(nbytes)``), host coder threads of ``pool``
    with the host ``tables`` below.  ``status``: a device decoder status checked before any file
    is written.  ``lock`` is held around the device coder call and the download of its streams
    (the device coder calls of one codec share scratch buffers), not around the file writes.
    Returns (bytes written, streams coded on the device)."""
    gn = len(paths)
    device_coded = 0
    if gn >= fe.GPU_CODER_MIN_STREAMS:
        with lock:
            packed, off = fe.encode_symbols_device(sym)
            host = pinned(packed.numel())
            host.copy_(packed, non_blocking=True)
            torch.cuda.current_stream(sym.device).synchronize()
        payload = host.numpy()
        device_coded = gn
    else:
        sym_h = sym.cpu().numpy()
        cdf, sz, offs = tables
        streams = list(pool.map(lambda k: encode_symbols(sym_h[k], cdf, sz, offs), range(gn)))
        off = np.zeros(gn + 1, dtype=np.int64)
        np.cumsum([len(s) for s in streams], out=off[1:])
        payload = np.frombuffer(b''.join(streams), dtype=np.uint8)
    if status is not None:
        fe.check_decode_status(status)
    hdr1 = np.frombuffer(struct.pack('>QQ', ps, ps), dtype=np.uint8)
    native_write(paths, np.broadcast_to(hdr1, (gn, 16)), payload, off, workers)
    return int(off[-1]) + 16 * gn, device_coded


def compress_tiles(tc, src, tiles, chunk_path, header_hw, workers, coder_tiles, stats,
                   device_source=None, level_arrays=None):
    """The 'cae' codec over ``tiles`` (list of (i, j) chunk indices) of the H x W x c uint8 slide
    ``src``: every tile is zero-padded to the full chunk, encoded, and written to
    ``chunk_path((i, j, 0))`` as '>QQ'(h, w) + rANS stream (R:549-555).

    ``device_source``: optional uint8 device tensor N x ps x ps x c holding the same tiles in
    order (inputs already resident in HBM: the device-resident measurement of bench.py).

    ``level_arrays``: optional ``DirArray`` of levels 1..K (``tiles`` must then be the whole
    slide in row-major order, read from ``src``; not with ``device_source``): every uploaded
    batch is also reduced into the levels (``region.PyramidWriter``) on the main stream after its
    encode; the level tiles are encoded in whole batches (``encode_level``, main stream) and coded
    through this call's coder workers.  Adds ``level_chunks`` and ``level_bytes`` to ``stats``."""
    if level_arrays and device_source is not None:
        raise ValueError('level_arrays: the levels are reduced from the uploaded source tiles, '
                         'not from device_source')
    H, W, c = src.shape if src is not None else (0, 0, tc.c_img)
    ps, B, dev = tc.ps, tc.batch, tc.dev
    fe = tc.fe
    n_tiles = len(tiles)
    tile_yx = np.ascontiguousarray(np.array(tiles, dtype=np.int32).reshape(-1, 2))
    pinned_src = device_source is None and _tiles_pinned(src, tile_yx, ps)
    L = C.lib()
    main = torch.cuda.current_stream(dev)
    s_in, s_code = tc.s_in, tc.s_code
    ev_up = [torch.cuda.Event() for _ in range(tc.slots)]
    ev_free = [None] * tc.slots
    stage = None
    if device_source is None and not pinned_src:
        stage = [tc.pinned('stage_in%d' % k, B * ps * ps * c).view(B, ps, ps, c) for k in range(2)]
        stage_ev = [None, None]
    sizes = group_sizes(n_tiles, coder_tiles, B)
    G = max(sizes)
    sym_all = [tc.buffer('sym_group%d' % k, (G, tc.cb, tc.lh * tc.lw), torch.int32)
               for k in range(2 if len(sizes) > 1 else 1)]
    coded = [None] * len(sym_all)       # per group buffer: (threading.Event, [cuda event]) of its job
    # two workers: the device coder calls are serialised by `code_lock` (they share scratch
    # buffers), but one group's chunk files are written while the next group is being coded
    coder = ThreadPoolExecutor(max_workers=2)
    code_lock = threading.Lock()
    jobs = []
    hdr1 = np.frombuffer(struct.pack('>QQ', *header_hw), dtype=np.uint8)
    pyr = None
    if level_arrays:
        from .region import PyramidWriter
        level_jobs = []
        level_lock = threading.Lock()         # one level group at a time: one streams buffer
        pool = ThreadPoolExecutor(max_workers=workers)       # host coder of small level groups
        tables = fe._host_tables()

        def code_level(sym, paths, ready):
            torch.cuda.set_device(dev)
            # code_lock around the device coder call only (as code_group): level-file writes do
            # not hold up the next level-0 coder call
            with level_lock, torch.cuda.stream(s_code):
                s_code.wait_event(ready)
                nbytes, _ = code_and_write(fe, tables, sym, paths, ps, workers,
                                           lambda n: tc.pinned('level_streams', n), pool,
                                           lock=code_lock)
                stats.add('level_bytes', nbytes)

        def level_group(sym, paths):
            ready = torch.cuda.Event()
            ready.record(main)
            level_jobs.append(coder.submit(code_level, sym, paths, ready))

        pyr = PyramidWriter((H, W, c), ps, len(level_arrays), B, dev,
                            lambda k, idx: level_arrays[k - 1].chunk_file(idx),
                            lambda run: tc.encode_level(len(run)), level_group,
                            (tc.cb, tc.lh * tc.lw), stage=tc.level_stage())
        stats['level_chunks'] = len(pyr.paths)
        stats['level_bytes'] = 0

    import time as _t
    t00 = _t.perf_counter()
    trace = stats.setdefault('trace', {}) if stats.get('want_trace') else None

    def mark(name):
        if trace is not None:
            trace[name] = round(_t.perf_counter() - t00, 4)

    def code_group(gi, lo, n, ready, launched, holder, before):
        torch.cuda.set_device(dev)
        if before is not None:
            before.result()              # the job that used this group's buffers last is done
        with code_lock, torch.cuda.stream(s_code):
            s_code.wait_event(ready)
            if trace is not None:
                ready.synchronize()
                mark('c_symbols_ready@%d' % lo)
            try:
                packed, off = fe.encode_symbols_device(sym_all[gi][:n])
                done = torch.cuda.Event()
                done.record(s_code)
                holder.append(done)          # the coder kernels have read the group buffer
            finally:
                launched.set()
            mark('c_coded@%d' % lo)
            host = tc.pinned('streams_out%d' % gi, packed.numel())
            host.copy_(packed, non_blocking=True)
            s_code.synchronize()
            mark('c_streams_on_host@%d' % lo)
        hdr = np.broadcast_to(hdr1, (n, 16))
        native_write([chunk_path((int(i), int(j), 0)) for i, j in tile_yx[lo:lo + n]], hdr,
                     host.numpy(), off, workers)
        mark('c_files_written@%d' % lo)
        stats.add('bytes', int(off[-1]) + 16 * n)
        stats.add('device_coded', n)

    gi, gpos, glo = 0, 0, 0
    for b, k0 in enumerate(range(0, n_tiles, B)):
        n = min(B, n_tiles - k0)
        slot = b % tc.slots
        if device_source is not None:
            x_dev = device_source[k0:k0 + n]
            if n == B and tc.graphs:
                tc.x[slot].copy_(x_dev, non_blocking=True)
                sym = tc.encode(slot, n)
            else:
                sym = tc.encode_eager(x_dev)
        else:
            with torch.cuda.stream(s_in):
                if ev_free[slot] is not None:
                    s_in.wait_event(ev_free[slot])
                if pinned_src:
                    band = tc.buffer('band_in%d' % slot, (B * ps * ps * c,), torch.uint8)
                    C.check(L.cae_tiles_upload_u8_banded(src.ctypes.data, H, W, c, ps,
                                                         tile_yx[k0:k0 + n].ctypes.data, n,
                                                         tc.x[slot].data_ptr(), band.data_ptr(),
                                                         _stream_ptr(s_in)))
                else:
                    sb = b & 1
                    if stage_ev[sb] is not None:
                        stage_ev[sb].synchronize()
                    native_gather(src, ps, tile_yx[k0:k0 + n], stage[sb].numpy()[:n], workers)
                    tc.x[slot][:n].copy_(stage[sb][:n], non_blocking=True)
                    stage_ev[sb] = torch.cuda.Event()
                    stage_ev[sb].record(s_in)
                ev_up[slot].record(s_in)
            main.wait_event(ev_up[slot])
            sym = tc.encode(slot, n)
            if pyr is not None:
                # on the main stream, before ev_free: the next upload into the slot waits for the
                # reduction; the upload stream waits for nothing else of the levels (DESIGN 3.5f)
                pyr.add(tc.x[slot], tile_yx[k0:k0 + n])
            ev_free[slot] = torch.cuda.Event()
            ev_free[slot].record(main)
        if gpos == 0 and coded[gi] is not None:
            launched, holder = coded[gi]
            launched.wait()
            if holder:
                main.wait_event(holder[0])       # the coder has consumed this group buffer
            coded[gi] = None
        sym_all[gi][gpos:gpos + n].copy_(sym.reshape(n, tc.cb, -1), non_blocking=True)
        gpos += n
        stats.add('pixels', n * ps * ps)
        if gpos >= sizes[len(jobs)] or k0 + n >= n_tiles:
            ready = torch.cuda.Event()
            ready.record(main)
            coded[gi] = (threading.Event(), [])
            jobs.append(coder.submit(code_group, gi, glo, gpos, ready, *coded[gi],
                                     jobs[-2] if len(jobs) >= 2 and len(sym_all) == 2 else None))
            glo += gpos
            gpos = 0
            gi = (gi + 1) % len(sym_all)
    if pyr is not None:
        pyr.finish()
    mark('c_all_batches_issued')
    for j in jobs + (level_jobs if pyr is not None else []):
        j.result()
    coder.shutdown()
    if pyr is not None:
        pool.shutdown()
    for st in (main, s_in, s_code):        # this call's streams only: another call may be in flight
        st.synchronize()
    mark('c_done')


def decompress_tiles(tc, tiles, chunk_path, workers, coder_tiles, stats, H, W, out_chunk_path=None,
                     out_image=None, device_sink=None):
    """Inverse of ``compress_tiles``: chunk files of ``tiles`` -> uint8 tiles, written as raw
    chunk files (``out_chunk_path``; the part of an edge chunk beyond the image is zero), or
    straight into the H x W x c host image ``out_image`` (page-locked for the copies to be
    asynchronous), or into ``device_sink`` (N x ps x ps x c uint8 on the device)."""
    ps, B, dev, c = tc.ps, tc.batch, tc.dev, tc.c_img
    fe = tc.fe
    n_tiles = len(tiles)
    tile_yx = np.ascontiguousarray(np.array(tiles, dtype=np.int32).reshape(-1, 2))
    L = C.lib()
    main = torch.cuda.current_stream(dev)
    s_out, s_code = tc.s_out, tc.s_dec
    sizes = group_sizes(n_tiles, coder_tiles, B)
    groups = [(int(sum(sizes[:k])), g) for k, g in enumerate(sizes)]
    reader = ThreadPoolExecutor(max_workers=1)
    tile_bytes = ps * ps * c
    out_pins = [tc.pinned('tiles_out%d' % k, B * tile_bytes).view(B, ps, ps, c)
                for k in range(tc.slots)] if out_chunk_path is not None else None
    writer = ThreadPoolExecutor(max_workers=2) if out_chunk_path is not None else None
    slot_busy = [None] * tc.slots          # D2H (and file write) still reading the slot's output
    wjobs = []
    expect_hdr = struct.pack('>QQ', ps, ps)
    import time as _t
    t00 = _t.perf_counter()
    trace = stats.setdefault('trace', {}) if stats.get('want_trace') else None

    def mark(name):
        if trace is not None:
            trace[name] = round(_t.perf_counter() - t00, 4)

    def load_group(gk):
        """chunk files -> pinned buffer -> device -> symbols (on the coder stream)."""
        lo, n = groups[gk]
        torch.cuda.set_device(dev)
        paths = [chunk_path((int(i), int(j), 0)) for i, j in tile_yx[lo:lo + n]]

        words = [None]

        def alloc(nbytes):
            words[0] = torch.empty((nbytes + 3) // 4, dtype=torch.int32, device=dev)
            if uploaded[gk & 1] is not None:
                uploaded[gk & 1].synchronize()       # the staging buffer's last upload has left it
            return tc.pinned('streams_in%d' % (gk & 1), nbytes).numpy()

        def upload(buf, lo, hi):
            # the streams of one run of files go up while the next run is read
            with torch.cuda.stream(s_code):
                words[0].view(torch.uint8)[lo:hi].copy_(torch.from_numpy(buf[lo:hi]), non_blocking=True)
                uploaded[gk & 1] = torch.cuda.Event()
                uploaded[gk & 1].record(s_code)
        with torch.cuda.stream(s_code):              # (the allocation belongs to the coder stream)
            hdr, payload, off = native_read(paths, 16, workers, alloc=alloc, slices=4, on_slice=upload)
        mark('d_files_read_g%d' % gk)
        if (off % 4).any() or bytes(hdr[0]) != expect_hdr or (hdr != hdr[0]).any():
            raise C.CaeError('chunk headers differ from the (patch, patch) the codec wrote')
        with torch.cuda.stream(s_code):
            # (no wait for the decoder here: this thread goes on to read the next group's files)
            sym, status = fe.decode_streams_device(words[0], off // 4, tc.lh * tc.lw, defer_status=True)
            statuses.append(status)
            done = torch.cuda.Event()
            done.record(s_code)
            if trace is not None:
                done.synchronize()
                mark('d_symbols_decoded_g%d' % gk)
        stats.add('device_decoded', n)
        return sym.reshape(n, tc.cb, tc.lh, tc.lw), done

    def write_batch(slot, k0, n, done):
        done.synchronize()
        img = out_pins[slot].numpy()
        for k in range(n):                        # zero what lies beyond the image (edge chunks)
            i, j = tile_yx[k0 + k]
            vh, vw = min(ps, H - i * ps), min(ps, W - j * ps)
            if vh < ps:
                img[k, vh:] = 0
            if vw < ps:
                img[k, :, vw:] = 0
        native_write([out_chunk_path((int(i), int(j), 0)) for i, j in tile_yx[k0:k0 + n]], None,
                     img.reshape(-1), np.arange(n + 1, dtype=np.int64) * tile_bytes, workers)

    statuses = []
    uploaded = [None, None]
    nxt = reader.submit(load_group, 0)
    b = 0
    for gk, (lo, gn) in enumerate(groups):
        sym, done = nxt.result()
        if gk + 1 < len(groups):
            nxt = reader.submit(load_group, gk + 1)
        main.wait_event(done)
        # allocated on the coder stream, read by this group's batches on the main stream: the
        # allocator must not hand the block to a later group's decoder before those have run
        sym.record_stream(main)
        for p0 in range(0, gn, B):
            n = min(B, gn - p0)
            slot = b % tc.slots
            b += 1
            if slot_busy[slot] is not None:
                busy = slot_busy[slot]
                if isinstance(busy, torch.cuda.Event):
                    main.wait_event(busy)
                else:
                    busy.result()                 # file write of the slot's previous batch
                    wjobs.remove(busy)
            if n == B and tc.graphs:
                tc.sym_in[slot].copy_(sym[p0:p0 + n], non_blocking=True)
                u8 = tc.decode(slot, n)
            else:
                u8 = tc.decode_eager(sym[p0:p0 + n])
            ev = torch.cuda.Event()
            ev.record(main)
            k0 = lo + p0
            for i, j in tile_yx[k0:k0 + n]:
                stats.add('pixels', int(min(ps, H - i * ps) * min(ps, W - j * ps)))
            if device_sink is not None:
                device_sink[k0:k0 + n].copy_(u8, non_blocking=True)
                continue
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev)
                if out_image is not None:
                    band = tc.buffer('band_out%d' % slot, (B * ps * ps * c,), torch.uint8)
                    C.check(L.cae_tiles_download_u8_banded(u8.data_ptr(), n, ps, c,
                                                           tile_yx[k0:k0 + n].ctypes.data,
                                                           out_image.ctypes.data, H, W,
                                                           band.data_ptr(), _stream_ptr(s_out)))
                    d = torch.cuda.Event()
                    d.record(s_out)
                    slot_busy[slot] = d
                else:
                    out_pins[slot][:n].copy_(u8, non_blocking=True)
                    d = torch.cuda.Event()
                    d.record(s_out)
                    job = writer.submit(write_batch, slot, k0, n, d)
                    wjobs.append(job)
                    slot_busy[slot] = job
            if not (n == B and tc.graphs):
                u8.record_stream(s_out)
    mark('d_all_batches_issued')
    if trace is not None:
        torch.cuda.synchronize(dev)
        mark('d_gpu_done')
    for j in list(wjobs):
        j.result()
    mark('d_files_written')
    reader.shutdown()
    if writer is not None:
        writer.shutdown()
    for st in (main, s_out, s_code):
        st.synchronize()
    for status in statuses:
        fe.check_decode_status(status)


def device_roundtrip(tc, x_dev, out_dev, coder_tiles):
    """The whole codec with every buffer resident in HBM (the device-resident measurement of
    ``bench.py``): uint8 tiles -> analysis transform + quantizer -> rANS streams of every tile
    (device coder, packed back to back) -> rANS decode -> de-quantizer + synthesis transform ->
    uint8 tiles, group by group on the current stream.  Returns the total stream bytes."""
    fe, B, dev = tc.fe, tc.batch, tc.dev
    n_tiles = x_dev.shape[0]
    G = max(B, min(coder_tiles, n_tiles))
    G = -(-G // B) * B
    sym_all = tc.buffer('sym_group0', (G, tc.cb, tc.lh * tc.lw), torch.int32)
    total = 0
    b = 0
    for lo in range(0, n_tiles, G):
        gn = min(G, n_tiles - lo)
        for p0 in range(0, gn, B):
            n = min(B, gn - p0)
            slot = b % tc.slots
            b += 1
            if n == B and tc.graphs:
                tc.x[slot].copy_(x_dev[lo + p0:lo + p0 + n], non_blocking=True)
                sym = tc.encode(slot, n)
            else:
                sym = tc.encode_eager(x_dev[lo + p0:lo + p0 + n])
            sym_all[p0:p0 + n].copy_(sym.reshape(n, tc.cb, -1), non_blocking=True)
        packed, off = fe.encode_symbols_device(sym_all[:gn])
        total += int(off[-1]) + 16 * gn
        sym2 = fe.decode_streams_device(packed.view(torch.int32), off // 4, tc.lh * tc.lw)
        sym2 = sym2.reshape(gn, tc.cb, tc.lh, tc.lw)
        for p0 in range(0, gn, B):
            n = min(B, gn - p0)
            slot = b % tc.slots
            b += 1
            if n == B and tc.graphs:
                tc.sym_in[slot].copy_(sym2[p0:p0 + n], non_blocking=True)
                u8 = tc.decode(slot, n)
            else:
                u8 = tc.decode_eager(sym2[p0:p0 + n])
            out_dev[lo + p0:lo + p0 + n].copy_(u8, non_blocking=True)
    return total


def phase_times(tc, x_dev, coder_tiles):
    """Device milliseconds of the four phases of one group (CUDA events on the current stream):
    analysis transforms + quantizer, rANS encode (+ scan / pack), rANS decode, de-quantizer +
    synthesis transforms.  For the per-phase record of bench.py."""
    fe, B, dev = tc.fe, tc.batch, tc.dev
    gn = min(x_dev.shape[0], max(B, coder_tiles)) // B * B
    if gn == 0:
        return None
    sym_all = torch.empty((gn, tc.cb, tc.lh * tc.lw), dtype=torch.int32, device=dev)
    out = torch.empty((gn, tc.ps, tc.ps, tc.c_img), dtype=torch.uint8, device=dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    torch.cuda.synchronize(dev)
    ev[0].record()
    for b, p0 in enumerate(range(0, gn, B)):
        slot = b % tc.slots
        if tc.graphs:
            tc.x[slot].copy_(x_dev[p0:p0 + B], non_blocking=True)
            sym = tc.encode(slot, B)
        else:
            sym = tc.encode_eager(x_dev[p0:p0 + B])
        sym_all[p0:p0 + B].copy_(sym.reshape(B, tc.cb, -1), non_blocking=True)
    ev[1].record()
    packed, off = fe.encode_symbols_device(sym_all)
    ev[2].record()
    sym2 = fe.decode_streams_device(packed.view(torch.int32), off // 4, tc.lh * tc.lw)
    sym2 = sym2.reshape(gn, tc.cb, tc.lh, tc.lw)
    ev[3].record()
    for b, p0 in enumerate(range(0, gn, B)):
        slot = b % tc.slots
        if tc.graphs:
            tc.sym_in[slot].copy_(sym2[p0:p0 + B], non_blocking=True)
            u8 = tc.decode(slot, B)
        else:
            u8 = tc.decode_eager(sym2[p0:p0 + B])
        out[p0:p0 + B].copy_(u8, non_blocking=True)
    ev[4].record()
    torch.cuda.synchronize(dev)
    names = ('analysis+quantize', 'rans_encode', 'rans_decode', 'dequantize+synthesis')
    rec = {n: round(ev[i].elapsed_time(ev[i + 1]), 3) for i, n in enumerate(names)}
    rec['chunks'] = gn
    rec['roundtrip_exact'] = bool(torch.equal(sym2.reshape(sym_all.shape), sym_all))
    return rec
