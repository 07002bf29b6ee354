#!/usr/bin/env python
"""Benchmark of the compress/decompress hot path (BASELINE.json metric: WSI encode+decode
megapixels per second at 1/2/4/8 B200, fraction of the tensor roofline, PSNR / bpp parity).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload wsi|patches|train] [--dump-outputs DIR]

Default workload ``wsi`` (BASELINE.json configs 3/4): a synthetic tissue-like whole-slide image
of 512 x 512 chunks, net A (3->128->128->48, level 3, LeakyReLU, random-init weights), sharded
over the N ranks by contiguous chunk range (``compress.shard_range``: 8192 chunks = 2.15
gigapixel per GPU -- a 50k x 50k slide is 9604 chunks -- no collective; the entropy coder's time
per call does not depend on the number of chunk streams, so it is handed the whole shard).  One *step* = the rank's shard through the public
``compress_image`` -> ``decompress_image`` (the reference's ``src/compress.py:29-128`` /
``src/decompress.py:40-96``), entropy coding included:

  e2e    host buffers: the slide lives in page-locked host memory, the chunk files (16-byte
         header + rANS stream each) are written to and read back from tmpfs, the reconstruction
         is written as raw chunk files; every H2D / D2H copy is inside the timed region;
  value  the same codec with the tiles resident in HBM when the clock starts: transforms,
         quantizer, rANS encode and decode of every chunk stream on the device, reconstruction
         left in HBM (``_slide.device_roundtrip``).

The line also carries: ``parity`` (symbol agreement, |dPSNR|, |d bpp| of sampled chunks against
the CPU oracle), ``roofline`` of the dominant kernel timed alone, ``device_resident_patches``
(the config-2 CUDA-graph replay of round 1, no entropy coding), ``cpu_baseline`` (the oracle on
this box's cores, bounded sample).  ``--workload patches`` is the round-1 bench (config 2) in
full; ``--workload train`` is the rate-distortion training step (config 5).

``--dump-outputs DIR`` (workload ``wsi``) writes what the last timed step of each region handed
its caller, so that two builds can be compared output for output on identical seeded inputs:
``DUMP_CHUNKS`` chunks of the reconstruction picked by a fixed seed (float32, N x 512 x 512 x 3,
uint8 values) from the e2e and the device-resident run, the stored bytes of each, the stored
chunk files (16-byte header + rANS stream, byte values as float32, back to back, with their
lengths) of the same chunks from the last step of the raw-chunk-file e2e variant, which keeps its
store, and the picked chunks' (row, column) indices (float64).
"""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ARCH_NAME = 'A'
BATCH, SIZE = 128, 256                  # config 2
PS, TILES, GX = 512, 8192, 64           # configs 3/4: chunk size, chunks per GPU, chunks per row
FLOPS_PER_PX = {'A': 136746, 'A_res': 321876, 'B': 367236, 'M': 738}   # SURVEY.md 8d
METRIC = 'wsi_encode_decode_megapixels_per_sec'
DUMP_CHUNKS = 8                         # 2 x 8 float32 chunks of 512 x 512 x 3 + streams: ~55 MB of dump
ARCH_TEXT = {'A': 'net A (3->128->128->48 L3 LeakyReLU)', 'A_res': 'net A+res',
             'B': 'net B (192 latent channels, L4, residual)'}


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(bf16=d['bf16_tflops'], bf16_sustained=d['bf16_tflops_sustained'],
                    hbm=d['hbm_gbs'], source='measured')
    return dict(bf16=1590.0, bf16_sustained=1400.0, hbm=6650.0, source='fallback')


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = ('timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None

    def window(self, t0, t1):
        self.t0, self.t1 = t0, t1

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                 '-i', str(self.index), '-lms', '25'], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        sm, mx, pw, reasons = [], [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        import datetime
        for r in self.rows:
            try:
                ts = datetime.datetime.strptime(r[0], '%Y/%m/%d %H:%M:%S.%f').timestamp()
                if self.t0 is not None and not (self.t0 - 0.05 <= ts <= self.t1 + 0.05):
                    continue
                r = r[1:]
                sm.append(float(r[0])); mx.append(float(r[1]))
                pw.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        return dict(sm_mhz=statistics.median(sm), sm_min_mhz=min(sm), sm_max_mhz=max(mx),
                    power_w_max=max(pw) if pw else None, reasons=sorted(reasons), samples=len(sm))


# ---------------------------------------------------------------------------------------------
# synthetic slide (configs 3/4)
# ---------------------------------------------------------------------------------------------
def slide_tile(O, i, j, ps=PS):
    """Chunk (i, j) of the synthetic slide: the oracle's tissue-like generator keyed on
    (i % 8, j % 8, seed 3), rolled by a chunk-dependent offset so that no two chunks are equal
    (cheap enough to fill gigapixels; reproducible by the parity check)."""
    import numpy as np
    bank = slide_tile.bank
    key = (i % 8, j % 8)
    if key not in bank:
        bank[key] = O.synth_tissue_tile(key[0], key[1], ps=ps, seed=3)
    return np.roll(bank[key], ((37 * i) % ps, (91 * j) % ps), axis=(0, 1))


slide_tile.bank = {}


def aligned_empty(nbytes, align=4096):
    import numpy as np
    raw = np.empty(nbytes + align, dtype=np.uint8)
    off = (-raw.ctypes.data) % align
    return raw[off:off + nbytes]


def wsi_workload_text(args, world):
    return (f'{ARCH_TEXT.get(args.arch, args.arch)}, synthetic tissue slide '
            f'{args.tiles * world // GX * PS}x{GX * PS}x3 uint8 in {PS}x{PS} chunks, '
            f'{args.tiles} chunks ({args.tiles * PS * PS / 1e9:.2f} GP) per GPU by contiguous chunk '
            f'range, compress_image -> decompress_image with rANS entropy coding')


def run_reference(args, rank, world):
    """The reference's CPU path for the same metric on a bounded sample: its own per-chunk codec
    flow (``ConvolutionalAutoencoder.encode`` / ``decode``, R:539-584: analysis transform at
    batch 1, quantize, rANS encode; rANS decode, synthesis transform, uint8) executed by the
    oracle restatement (bit-exact against the reference classes; the CompressAI pieces restated),
    fp32, all host threads."""
    if rank != 0:
        return
    import torch
    from oracle import cae_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    chk = O.make_checkpoint(O.NAMED_ARCHS[args.arch], seed=1234)
    model = O.OracleModel(chk)
    if args.workload == 'patches':
        n = 8
        x_u8 = O.synth_natural(n, 3, SIZE, SIZE, seed=1)

        def step():
            x = x_u8.float() / 255.0
            out = model.forward(x)
            O.rate_loss(x, out['p_y'])
            (out['x_r'][0] * 255.0).clip(0, 255).to(torch.uint8)
        px = n * SIZE * SIZE
        sample = f'{n} of {BATCH} tiles of {SIZE}x{SIZE} per step (CPU fp32, torch {torch.__version__})'
        workload = (f'{ARCH_TEXT.get(args.arch, args.arch)}, {BATCH}x3x{SIZE}x{SIZE} uint8 patches per GPU, '
                    'encode+quantize+rate+decode')
    else:
        n = 2
        tiles = [slide_tile(O, 0, j) for j in range(n)]

        def step():
            for t in tiles:
                blob = model.codec_encode(t)
                model.codec_decode(blob)
        px = n * PS * PS
        sample = (f'{n} of {args.tiles} chunks of {PS}x{PS} per step, one chunk at a time like the '
                  f"reference's codec (CPU fp32, torch {torch.__version__}, C rANS)")
        workload = wsi_workload_text(args, world)
    for _ in range(max(1, min(args.warmup, 2))):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    val = px * args.steps / 1e6 / dt
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': round(val, 4), 'unit': 'MP/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': round(dt / args.steps * 1e3, 3), 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': workload, 'sample': sample,
                   'note': 'value is a per-pixel rate of the bounded sample, comparable with the '
                           'GPU arm\'s MP/s'},
        'cpu_baseline': {'value': round(val, 4), 'unit': 'MP/s', 'cores': cores, 'kind': 'port',
                         'sample': sample},
        'e2e': {'value': round(val, 4), 'unit': 'MP/s', 'h2d_bytes_per_step': 0,
                'd2h_bytes_per_step': 0}}))


# ---------------------------------------------------------------------------------------------
# shared pieces
# ---------------------------------------------------------------------------------------------
class Ctx:
    pass


def setup(args):
    import torch
    import torch.distributed as dist
    c = Ctx()
    c.rank = int(os.environ.get('RANK', 0))
    c.world = int(os.environ.get('WORLD_SIZE', 1))
    c.local = int(os.environ.get('LOCAL_RANK', 0))
    if not torch.cuda.is_available():
        sys.exit('bench.py: no CUDA device (the hot path has no CPU fallback)')
    torch.cuda.set_device(c.local)
    if c.world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', c.local))
    c.flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')   # > 126 MB L2

    def flush_l2():
        # write 256 MiB (evicts everything), then read it back so the L2 is left holding
        # clean lines: otherwise the first timed kernel pays for writing back the fill
        c.flush.fill_(1)
        c.flush.view(torch.int64).sum()

    def barrier():
        torch.cuda.synchronize()
        if c.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device='cuda')
        if c.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    def sum_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device='cuda')
        if c.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return t.item()
    c.flush_l2, c.barrier, c.max_over_ranks, c.sum_over_ranks = flush_l2, barrier, max_over_ranks, sum_over_ranks
    return c


def dominant_kernel_roofline(c, model, x_u8_dev, peaks, traffic=None):
    """The 128->128 stride-1 implicit-GEMM layer timed ALONE (one launch between
    synchronisations, L2 flush queued right before it), against the measured bf16 peaks."""
    import torch
    from cnn_autoencoder_b200 import _cabi, _ops
    with torch.no_grad():
        model['encoder'](x_u8_dev)                # eager: records the ABI calls of every layer
    ex = model['encoder'].module._executor()
    dom = None
    for k, st in enumerate(ex.steps):
        if st.kind == _cabi.CONV_S1 and st.c_in >= 64:
            dom = k
            break
    if dom is None or dom not in ex.last_calls:
        return None
    call = ex.last_calls[dom]
    # MEASURED_PEAKS.json's burst figure is a best-of-10 on a device that was not under sustained
    # load: give this kernel the same footing by letting the device idle for a moment first
    torch.cuda.synchronize()
    time.sleep(2.0)
    for _ in range(3):
        _ops.replay(call)
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
           for _ in range(20)]
    for s, e in evs:
        c.flush_l2()
        s.record()
        _ops.replay(call)
        e.record()
        torch.cuda.synchronize()
    times = sorted(s.elapsed_time(e) for s, e in evs)
    t_ms = statistics.mean(times)            # the average launch, as the contract asks
    x_in = call[0][1]
    st = ex.steps[dom]
    flops = 2.0 * 9 * st.c_in * st.c_out * x_in.n * x_in.h * x_in.w
    ach = flops / (t_ms / 1e3) / 1e12
    return {'bound': 'tensor', 'achieved': round(ach, 2), 'peak': peaks['bf16'],
            'unit': 'TFLOP/s', 'frac': round(ach / peaks['bf16'], 4),
            'frac_of_sustained_peak': round(ach / peaks['bf16_sustained'], 4),
            'peak_sustained': peaks['bf16_sustained'],
            # dram__bytes_read.sum + dram__bytes_write.sum of one launch of this shape, a constant
            # copied from the committed ncu --set full capture (profiles/), not measured per run
            'traffic': traffic, 'traffic_source': 'profiles/r02_ncu_step.csv row 2: dram__bytes_read.sum + dram__bytes_write.sum of one '
                              'ncu --set full capture of this kernel at this shape (a constant, not re-measured per run)',
            'kernel': 'igemm_conv_kernel<EPI_ACT> conv3x3 s1 %d->%d @%dx%d x%d' % (
                st.c_in, st.c_out, x_in.h, x_in.w, x_in.n),
            'algorithmic_flops_per_launch': flops,
            'ms': round(t_ms, 4), 'ms_median': round(statistics.median(times), 4),
            'ms_min': round(times[0], 4), 'ms_max': round(times[-1], 4),
            'peak_source': peaks['source'] + ' bf16 burst (frac) and sustained'}


def patches_device_resident(c, args, model, O, steps, warmup):
    """Config 2: 128 x 3 x 256 x 256 uint8 patches resident in HBM, encode + quantize + rate +
    decode as one CUDA-graph replay per step (no entropy coding).  Returns a dict."""
    import torch
    from cnn_autoencoder_b200.pipeline import CodecPipeline
    pipe = CodecPipeline(model)
    B = args.batch
    x_host = O.synth_natural(B, 3, SIZE, SIZE, seed=1 + c.rank).permute(0, 2, 3, 1).contiguous()
    x_dev = x_host.pin_memory().cuda(non_blocking=True)
    graph = None
    if not args.no_graph:
        try:
            graph = pipe.graphed(x_dev, warmup=warmup)
        except RuntimeError as exc:
            print(f'bench.py: CUDA graph capture failed ({exc}); timing eager launches', file=sys.stderr)
    run = graph.replay if graph is not None else (lambda: pipe(x_dev))
    for _ in range(warmup):
        out = run()
    c.barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(steps)]
    for s, e in ev:
        c.flush_l2()
        s.record()
        out = run()
        e.record()
    c.barrier()
    total_ms = c.max_over_ranks(sum(s.elapsed_time(e) for s, e in ev))
    px = B * SIZE * SIZE
    value = c.world * px * steps / (total_ms / 1e3) / 1e6
    return dict(value=round(value, 2), unit='MP/s', ms_per_step=round(total_ms / steps, 4),
                steps=steps, est_bpp=round(out['bpp'].item(), 4),
                launches_per_step=graph.launches if graph is not None else None,
                workload=f'{B}x3x{SIZE}x{SIZE} uint8 patches per GPU resident in HBM, encode+quantize+'
                         'rate+decode, one CUDA graph replay per step, L2 flushed between steps',
                tflops=round(value * 1e6 * FLOPS_PER_PX[args.arch] / 1e12 / c.world, 2)), x_dev


# ---------------------------------------------------------------------------------------------
# workload: WSI (configs 3/4) -- the default
# ---------------------------------------------------------------------------------------------
def run_wsi(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from oracle import cae_oracle as O       # weights / tiles generator + parity + cpu_baseline only
    import cnn_autoencoder_b200 as M
    from concurrent.futures import ThreadPoolExecutor
    from cnn_autoencoder_b200 import _cabi, _slide, _store
    from cnn_autoencoder_b200 import compress as CMP
    from cnn_autoencoder_b200 import decompress as DEC
    from cnn_autoencoder_b200._entropy import decode_symbols
    from cnn_autoencoder_b200._store import DirArray
    from cnn_autoencoder_b200.jobs import SlideJobs

    c = setup(args)
    rank, world = c.rank, c.world
    warmup = max(args.warmup, 3)
    peaks = measured_peaks()
    arch = O.NAMED_ARCHS[args.arch]
    chk = O.make_checkpoint(arch, seed=1234)
    model = CMP.load_model(chk)
    level = len(model['encoder'].module.analysis_track)

    # ---- the slide: GX chunks per row, tiles*world chunks in all; this rank's rows only are
    # touched (and page-locked): shard_range hands rank k the k-th contiguous range
    T = args.tiles
    if T % GX:
        sys.exit(f'--tiles must be a multiple of {GX}')
    rows_per_rank = T // GX
    H, W = rows_per_rank * world * PS, GX * PS
    row_bytes = PS * W * 3
    slide = aligned_empty(H * W * 3).reshape(H, W, 3)        # virtual: untouched rows cost nothing
    mine = slide[rank * rows_per_rank * PS:(rank + 1) * rows_per_rank * PS]
    t_gen = time.perf_counter()
    for i in range(rank * rows_per_rank, (rank + 1) * rows_per_rank):
        for j in range(GX):
            slide[i * PS:(i + 1) * PS, j * PS:(j + 1) * PS] = slide_tile(O, i, j)
    t_gen = time.perf_counter() - t_gen
    pin = _slide.pin_array(mine)
    # the reconstruction goes straight into a caller-owned array of the slide's shape (this
    # rank's rows page-locked, like the source)
    recon = aligned_empty(H * W * 3).reshape(H, W, 3)
    recon_mine = recon[rank * rows_per_rank * PS:(rank + 1) * rows_per_rank * PS]
    recon_mine[:] = 0
    pin_r = _slide.pin_array(recon_mine)
    base = '/dev/shm' if os.path.isdir('/dev/shm') and shutil.disk_usage('/dev/shm').free > 8 * H * W else '/tmp'
    tag = os.environ.get('MASTER_PORT', str(os.getpid()))
    work = os.path.join(base, f'cae_bench_{tag}')
    if rank == 0:
        shutil.rmtree(work, ignore_errors=True)
        os.makedirs(work, exist_ok=True)
    c.barrier()

    if args.coder_tiles <= 0:
        args.coder_tiles = T
    def schedule(text):
        v = [int(x) for x in str(text).split(',') if x.strip()]
        return v[0] if len(v) == 1 else v

    # coder groups of the e2e step: the tile loops' own default (`_slide.default_schedule`) unless named
    args.e2e_coder_tiles = schedule(args.e2e_coder_tiles) or _slide.default_schedule(T, args.batch_tiles)
    args.e2e_decoder_tiles = (schedule(args.e2e_decoder_tiles) or
                              _slide.default_schedule(T, args.batch_tiles, decode=True))
    kw = dict(rank=rank, world_size=world, batch_tiles=args.batch_tiles)

    # Every step compresses into a store of its own, as a job that works through a list of slides
    # does (a chunk file renamed over last step's file frees that file's pages inside the rename:
    # 57 ms instead of 21 ms per 4096 chunk files on this tmpfs, tools/micro/filebench.cpp).  Two
    # stores alternate; a rank unlinks its own chunk files of step k on a background thread once
    # step k has been decompressed (inside the timed region); rank 0 removes what is left at the end.
    #
    # The steps of the timed region are in flight two at a time (`jobs.SlideJobs`): the
    # compress_image call of step k + 1 runs beside the decompress_image call of step k, each on
    # its own thread and CUDA stream -- what a job working through a list of slides does with the
    # two directions of the host link and with the GPU time under one call's tail and the other's
    # prologue.  Every call, copy and file operation of the K steps lies inside the timed region;
    # `e2e.one_step_at_a_time` is the same measured with the calls strictly one after the other.
    my_chunks = [(i, j, 0) for i in range(rank * rows_per_rank, (rank + 1) * rows_per_rank) for j in range(GX)]
    dump = {} if args.dump_outputs and rank == 0 else None
    dump_yx = [my_chunks[k][:2] for k in sorted(np.random.default_rng(0).choice(T, DUMP_CHUNKS, replace=False))]
    cleaner = ThreadPoolExecutor(max_workers=1)
    jobs = SlideJobs(c.local)
    state = dict(step=0, dec={}, clean={})

    def remove_chunks(root, group):
        d = os.path.join(root, group)
        _store.native_remove([os.path.join(d, '.'.join(map(str, idx))) for idx in my_chunks], 4)

    def stores(k):
        return tuple(os.path.join(work, f'{name}_{k % 2}.zarr') for name in ('slide', 'recon'))

    def compress_job(k):
        for waits in (state['dec'], state['clean']):       # the store of step k - 2 is empty again
            if k - 2 in waits:
                waits.pop(k - 2).result()
        cs = CMP.compress_image('CAE', chk, slide, stores(k)[0], patch_size=PS, gpu=True,
                                coder_tiles=args.e2e_coder_tiles, **kw)
        cs['store'] = stores(k)[0]
        return cs

    def decompress_job(k, compressed, to_files, keep):
        cs = compressed.result()
        comp_dir, recon_dir = stores(k)
        ds = DEC.decompress_image(comp_dir, recon_dir if to_files else recon, checkpoint=chk,
                                  gpu=True, coder_tiles=args.e2e_decoder_tiles, **kw)
        if not keep:
            last = [(comp_dir, '0/0')] + ([(recon_dir, 'decompressed/0/0')] if to_files else [])
            state['clean'][k] = cleaner.submit(lambda: [remove_chunks(*a) for a in last])
        return cs, ds

    def run(n, to_files=False, keep_last=False):
        """n steps, at most two in flight; returns [(compress stats, decompress stats)]."""
        futs = []
        for i in range(n):
            k = state['step']
            state['step'] += 1
            fc = jobs.submit('compress', compress_job, k)
            fd = jobs.submit('decompress', decompress_job, k, fc, to_files, keep_last and i == n - 1)
            state['dec'][k] = fd
            futs.append(fd)
        return [f.result(timeout=300) for f in futs]       # (a hang becomes an error, not a dead box)

    def timed(fn):
        """(device ms, wall s) of fn() between two idle points of the device, max over ranks."""
        torch.cuda.synchronize()
        c.barrier()
        s0, e0 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        w0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()          # every stream of every call
        e0.record()
        e0.synchronize()
        c.barrier()
        return out, c.max_over_ranks(s0.elapsed_time(e0)), time.perf_counter() - w0

    # ---- e2e: host buffers, files on tmpfs, copies inside ----
    for _ in range(warmup):
        (cs, ds), = run(1)
    assert cs.get('engine') == 'slide' and ds.get('engine') == 'slide', 'tile loops fell off the batched engine'
    if args.e2e_in_flight > 1:
        run(2)
    tc = _slide.tile_codec(model, PS, 3, args.batch_tiles)
    c.barrier()
    phases = {}
    with ClockSampler(c.local) as clk:
        time.sleep(0.3)
        launches0, replays0 = _cabi.launch_count(), (tc.replays_enc, tc.replays_dec)
        t_begin = time.time()
        if args.e2e_in_flight > 1:
            try:
                done, e2e_ms, wall = timed(lambda: run(args.steps))
            except Exception as exc:       # report the one-at-a-time figure rather than nothing
                print(f'WARNING: two steps in flight failed ({exc!r}); measuring one step at a time',
                      file=sys.stderr)
                args.e2e_in_flight = 1
                jobs.close(wait=False)
                jobs = SlideJobs(c.local)
                state.update(step=state['step'] + 2, dec={}, clean={})
        if args.e2e_in_flight == 1:
            done, e2e_ms, wall = timed(lambda: [run(1)[0] for _ in range(args.steps)])
        if dump is not None:      # taken now: the variants below write the reconstruction again
            dump['e2e_reconstruction'] = np.stack([recon[i * PS:(i + 1) * PS, j * PS:(j + 1) * PS]
                                                   for i, j in dump_yx]).astype(np.float32)
            dump['e2e_stored_bytes'] = np.array([done[-1][0]['bytes']], np.float64)
        for cs, ds in done:
            for k, v in (('compress_s', cs['seconds']), ('decompress_s', ds['seconds'])):
                phases[k] = phases.get(k, 0.0) + v
        clk_e2e_window = (t_begin, time.time())
        launches_e2e = (_cabi.launch_count() - launches0 +
                        (tc.replays_enc - replays0[0]) * tc.launches_enc +
                        (tc.replays_dec - replays0[1]) * tc.launches_dec)
        px_step = T * PS * PS
        e2e_value = world * px_step * args.steps / (e2e_ms / 1e3) / 1e6
        # the same with one call after the other (2 steps)
        seq, seq_ms, _ = timed(lambda: [run(1)[0] for _ in range(2)])
        e2e_seq = {'value': round(world * px_step * 2 / (seq_ms / 1e3) / 1e6, 2), 'unit': 'MP/s', 'steps': 2,
                   'ms_per_step': round(seq_ms / 2, 3),
                   'compress_s': round(sum(a['seconds'] for a, _ in seq) / 2, 4),
                   'decompress_s': round(sum(b['seconds'] for _, b in seq) / 2, 4)}
        # variant: the reconstruction written as raw chunk files on tmpfs (2 steps, reported aside)
        run(1, to_files=True)
        files, files_ms, _ = timed(lambda: [run(1, to_files=True, keep_last=(i == 1))[0] for i in range(2)])
        cs, ds = files[-1]
        e2e_files_value = world * px_step * 2 / (files_ms / 1e3) / 1e6
        stored = DirArray(os.path.join(cs['store'], '0/0'), mode='r')       # the last step's store is kept
        if dump is not None:      # what compress_image stored for the sampled chunks: header + rANS stream
            streams = [np.frombuffer(stored.read_encoded((i, j, 0)), np.uint8) for i, j in dump_yx]
            dump['e2e_chunk_streams'] = np.concatenate(streams).astype(np.float32)
            dump['e2e_chunk_stream_bytes'] = np.array([s.size for s in streams], np.float64)
        comp_bytes_rank = cs['bytes']

        # ---- value: the same codec, everything resident in HBM ----
        x_dev = torch.empty((T, PS, PS, 3), dtype=torch.uint8, device='cuda')
        tiles_mine = [(i, j) for i in range(rank * rows_per_rank, (rank + 1) * rows_per_rank) for j in range(GX)]
        yx = np.array(tiles_mine, dtype=np.int32)
        for k0 in range(0, T, 256):
            _cabi.check(_cabi.lib().cae_tiles_upload_u8(slide.ctypes.data, H, W, 3, PS,
                                                        yx[k0:k0 + 256].ctypes.data, min(256, T - k0),
                                                        x_dev[k0:].data_ptr(), None))
        torch.cuda.synchronize()
        out_dev = torch.empty_like(x_dev)
        for _ in range(warmup):
            _slide.device_roundtrip(tc, x_dev, out_dev, args.coder_tiles)
        c.barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
              for _ in range(args.steps)]
        launches0, replays0 = _cabi.launch_count(), (tc.replays_enc, tc.replays_dec)
        t_begin = time.time()
        for s, e in ev:
            s.record()
            stored_bytes = _slide.device_roundtrip(tc, x_dev, out_dev, args.coder_tiles)
            e.record()
        c.barrier()
        clk.window(t_begin, time.time())
        launches = (_cabi.launch_count() - launches0 + (tc.replays_enc - replays0[0]) * tc.launches_enc +
                    (tc.replays_dec - replays0[1]) * tc.launches_dec)
        total_ms = c.max_over_ranks(sum(s.elapsed_time(e) for s, e in ev))
        value = world * px_step * args.steps / (total_ms / 1e3) / 1e6
        if dump is not None:
            k = [(i - rank * rows_per_rank) * GX + j for i, j in dump_yx]
            dump['device_reconstruction'] = out_dev[k].cpu().numpy().astype(np.float32)
            dump['device_stored_bytes'] = np.array([stored_bytes], np.float64)
    clocks = clk.summary()
    clk.window(*clk_e2e_window)
    clocks_e2e = clk.summary()

    # ---- the reconstruction the e2e calls left in host memory against the device-resident run's
    # (same kernels, and the coder is lossless: identical bytes expected), 64 sampled chunks ----
    torch.cuda.synchronize()
    same_tiles = 0
    sample = [tiles_mine[(k * 131) % T] for k in range(64)]
    for (i, j) in sample:
        got = recon[i * PS:(i + 1) * PS, j * PS:(j + 1) * PS]
        ref = out_dev[(i - rank * rows_per_rank) * GX + j].cpu().numpy()
        same_tiles += int(np.array_equal(got, ref))
    e2e_matches_device = {'chunks': len(sample), 'identical': same_tiles}
    if same_tiles != len(sample):
        print(f'WARNING: e2e reconstruction differs from the device-resident run: {e2e_matches_device}',
              file=sys.stderr)

    # ---- per-phase device times of one step (events around each phase, rank 0) ----
    per_phase = _slide.phase_times(tc, x_dev[:min(T, args.coder_tiles)], args.coder_tiles)

    # ---- parity gates: sampled chunks against the CPU oracle (rank 0) ----
    parity = None
    if rank == 0 and not args.no_parity:
        torch.set_num_threads(os.cpu_count() or 1)
        om = O.OracleModel(chk)
        fe = model['fact_ent'].module
        cdf, sizes, offs = fe._host_tables()
        lh = PS // 2 ** level
        idx = [tiles_mine[(k * 997) % T] for k in range(args.parity_tiles)]
        agree = n_sym = 0
        max_frac = 0.0
        sse_p = sse_o = 0.0
        bits_p = bits_o = 0.0
        for (i, j) in idx:
            tile = slide[i * PS:(i + 1) * PS, j * PS:(j + 1) * PS]
            ref = om.codec_trace(tile)       # y, symbols, p of symbols, x_r uint8 (oracle, fp32 CPU)
            raw = stored.read_encoded((i, j, 0))
            sym = decode_symbols(raw[16:], fe.channels, lh * lh, cdf, sizes, offs).reshape(fe.channels, lh, lh)
            sym_o = ref['symbols'].numpy().reshape(sym.shape)
            same = sym == sym_o
            agree += int(same.sum()); n_sym += sym.size
            if not same.all():
                # flipped symbols must sit at a rounding boundary of the oracle's latent
                yv = ref['y_minus_median'].numpy().reshape(sym.shape)[~same]
                max_frac = max(max_frac, float(np.abs(np.abs(yv - np.floor(yv)) - 0.5).max()))
            bits_p += float(om.symbol_bits(torch.from_numpy(sym.astype(np.int32))))
            bits_o += float(om.symbol_bits(ref['symbols']))
            rec = recon[i * PS:(i + 1) * PS, j * PS:(j + 1) * PS].astype(np.float64)
            sse_p += float(((rec - tile.astype(np.float64)) ** 2).sum())
            sse_o += float(((ref['x_r_u8'].astype(np.float64) - tile.astype(np.float64)) ** 2).sum())
        npx = len(idx) * PS * PS
        psnr = lambda sse: 20 * np.log10(255.0) - 10 * np.log10(max(sse, 1e-12) / (npx * 3))
        parity = {'chunks': len(idx), 'symbol_agreement_pct': round(100.0 * agree / n_sym, 5),
                  'max_distance_of_a_flip_from_a_rounding_boundary': round(max_frac, 5),
                  'psnr_db': round(float(psnr(sse_p)), 4), 'oracle_psnr_db': round(float(psnr(sse_o)), 4),
                  'abs_dpsnr_db': round(abs(float(psnr(sse_p) - psnr(sse_o))), 5),
                  'est_bpp': round(bits_p / npx, 5), 'oracle_est_bpp': round(bits_o / npx, 5),
                  'abs_dbpp_pct': round(100.0 * abs(bits_p - bits_o) / bits_o, 5),
                  'gates': 'agreement >= 99.9 %, |dPSNR| <= 0.05 dB, |d bpp| <= 0.5 % (north star)'}
        parity['pass'] = bool(parity['symbol_agreement_pct'] >= 99.9 and parity['abs_dpsnr_db'] <= 0.05
                              and parity['abs_dbpp_pct'] <= 0.5)

    # ---- config 2 sub-record + roofline of the dominant kernel (rank 0 for the roofline) ----
    sub, x_patch = patches_device_resident(c, args, model, O, steps=min(args.steps, 20), warmup=3)
    stored_bpp = 8.0 * c.sum_over_ranks(comp_bytes_rank) / (world * px_step)
    if rank != 0:
        pin.close()
        pin_r.close()
        if world > 1:
            dist.destroy_process_group()
        return
    roof = dominant_kernel_roofline(c, model, tc.x[0], peaks,
                                    traffic=1119336448 if args.batch_tiles * 4 == BATCH else None)

    # ---- CPU baseline (bounded sample, rank 0, N = 1 only) ----
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        om = O.OracleModel(chk)
        tiles = [slide_tile(O, 0, j) for j in range(2)]
        om.codec_decode(om.codec_encode(tiles[0]))
        t0 = time.perf_counter()
        reps = 2
        for _ in range(reps):
            for t in tiles:
                om.codec_decode(om.codec_encode(t))
        dt = (time.perf_counter() - t0) / reps
        cpu = {'value': round(len(tiles) * PS * PS / 1e6 / dt, 4), 'unit': 'MP/s', 'cores': cores,
               'kind': 'port',
               'sample': f'{len(tiles)} of {T} chunks of {PS}x{PS}, one chunk at a time like the reference\'s '
                         f'codec, {reps} repeats after 1 warm-up (oracle: reference transforms restated + '
                         'restated EntropyBottleneck + C rANS)'}

    tf = value * 1e6 * FLOPS_PER_PX[args.arch] / 1e12 / world
    line = {
        'metric': METRIC, 'value': round(value, 2), 'unit': 'MP/s', 'n_gpus': world,
        'steps': args.steps, 'warmup': warmup, 'ms_per_step': round(total_ms / args.steps, 3),
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f16',
        'data': 'synthetic',
        'config': {'workload': wsi_workload_text(args, world),
                   'l2': f'inputs larger than L2 ({px_step * 3 / 1e9:.2f} GB of tiles per step per GPU)',
                   'accumulate': 'f32', 'batch_tiles': args.batch_tiles, 'coder_tiles': args.coder_tiles,
                   'e2e_coder_tiles': args.e2e_coder_tiles, 'e2e_decoder_tiles': args.e2e_decoder_tiles,
                   'value_is': 'tiles resident in HBM -> transforms + quantizer + device rANS encode + '
                               'decode + transforms -> tiles in HBM (no host transfer)',
                   'e2e_is': 'compress_image -> decompress_image: slide in page-locked host memory -> chunk '
                             f'files (header + rANS stream) on {base} -> reconstruction in page-locked host '
                             'memory; every H2D / D2H copy and file write / read inside the timed region; '
                             'each step writes a store of its own (two alternate; a step\'s chunk files are '
                             'unlinked by a background thread inside the timed region once it has been '
                             'decompressed)' + ('; two steps in flight: the compress_image call of step k + 1 '
                             'runs beside the decompress_image call of step k, each on its own thread and CUDA '
                             'stream (jobs.SlideJobs) -- all calls of the K steps start and end inside the timed '
                             'region; e2e.one_step_at_a_time is the same with the calls one after the other'
                             if args.e2e_in_flight > 1 else ''),
                   'e2e_steps_in_flight': args.e2e_in_flight,
                   'timed_region_s': {'value': round(total_ms / 1e3, 3), 'e2e': round(e2e_ms / 1e3, 3)},
                   'stored_bpp': round(stored_bpp, 4), 'slide_generation_s': round(t_gen, 1)},
        'clocks': clocks, 'clocks_e2e': clocks_e2e,
        'e2e': {'value': round(e2e_value, 2), 'unit': 'MP/s',
                'h2d_bytes_per_step': int(px_step * 3 + comp_bytes_rank),
                'd2h_bytes_per_step': int(px_step * 3 + comp_bytes_rank),
                'ms_per_step': round(e2e_ms / args.steps, 3), 'wall_s': round(wall, 3),
                'phase_s_per_step': {k: round(v / args.steps, 4) for k, v in phases.items()},
                'gpu_launches': int(launches_e2e),
                'one_step_at_a_time': e2e_seq,
                'reconstruction_vs_device_resident_run': e2e_matches_device,
                'with_reconstruction_written_as_raw_chunk_files': {
                    'value': round(e2e_files_value, 2), 'unit': 'MP/s', 'steps': 2,
                    'one_step_at_a_time': True}},
        'gpu_launches': int(launches),
        'device_phase_ms': per_phase,
        'pipeline_tflops': round(tf, 2),
        'pipeline_tensor_frac': round(tf / peaks['bf16'], 4),
        'pipeline_tensor_frac_of_sustained_peak': round(tf / peaks['bf16_sustained'], 4),
        'parity': parity, 'device_resident_patches': sub,
        'roofline': roof, 'cpu_baseline': cpu,
    }
    if dump is not None:
        dump['chunks'] = np.array(dump_yx, np.float64)
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, name + '.npy'), a)
    print(json.dumps(line))
    pin.close()
    pin_r.close()
    shutil.rmtree(work, ignore_errors=True)
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------
# workload: patches (config 2) -- the round-1 bench
# ---------------------------------------------------------------------------------------------
def run_patches(args):
    import torch
    import torch.distributed as dist
    from oracle import cae_oracle as O
    import cnn_autoencoder_b200 as M
    from cnn_autoencoder_b200.pipeline import CodecPipeline

    c = setup(args)
    rank, world = c.rank, c.world
    warmup = max(args.warmup, 3)
    peaks = measured_peaks()
    chk = O.make_checkpoint(O.NAMED_ARCHS[args.arch], seed=1234)
    model = M.autoencoder_from_state_dict(chk, gpu=True, train=False)
    with ClockSampler(c.local) as clk:
        time.sleep(0.4)
        t_begin = time.time()
        sub, x_dev = patches_device_resident(c, args, model, O, steps=args.steps, warmup=warmup)
        clk.window(t_begin, time.time())
    B = args.batch
    px_per_step = B * SIZE * SIZE

    # end to end through CodecPipeline from pinned host buffers (H2D / D2H inside)
    pipe = CodecPipeline(model)
    x_pin = x_dev.cpu().pin_memory()
    main = torch.cuda.current_stream()
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    x_stage = [torch.empty_like(x_dev) for _ in range(2)]
    out_stage = [torch.empty_like(x_pin).pin_memory() for _ in range(2)]
    bpp_stage = [torch.empty(1, dtype=torch.float64).pin_memory() for _ in range(2)]
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_free = [torch.cuda.Event() for _ in range(2)]
    ev_done = [torch.cuda.Event() for _ in range(2)]
    ev_out = [torch.cuda.Event() for _ in range(2)]
    g_e2e = None if args.no_graph else [pipe.graphed(x_stage[k]) for k in range(2)]

    def e2e_run(n_steps):
        for i in range(n_steps):
            k = i % 2
            with torch.cuda.stream(s_in):
                if i >= 2:
                    s_in.wait_event(ev_free[k])
                x_stage[k].copy_(x_pin, non_blocking=True)
                ev_in[k].record(s_in)
            main.wait_event(ev_in[k])
            if g_e2e is None:
                o = pipe(x_stage[k])
            else:
                if i >= 2:
                    main.wait_event(ev_out[k])
                o = g_e2e[k].replay()
            ev_free[k].record(main)
            ev_done[k].record(main)
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_done[k])
                if g_e2e is None:
                    o['x_r_u8'].record_stream(s_out)
                    o['bpp'].record_stream(s_out)
                out_stage[k].copy_(o['x_r_u8'], non_blocking=True)
                bpp_stage[k].copy_(o['bpp'], non_blocking=True)
                ev_out[k].record(s_out)
        s_out.synchronize()
        s_in.synchronize()

    e2e_run(3)
    c.barrier()
    s0, e0 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    e2e_run(args.steps)
    main.wait_stream(s_out)
    e0.record()
    c.barrier()
    e2e_ms = c.max_over_ranks(s0.elapsed_time(e0))
    e2e_value = world * px_per_step * args.steps / (e2e_ms / 1e3) / 1e6
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    roof = dominant_kernel_roofline(c, model, x_dev, peaks,
                                    traffic=1119336448 if (B == BATCH and args.arch == ARCH_NAME) else None)
    line = {
        'metric': 'patch_encode_decode_megapixels_per_sec', 'value': sub['value'], 'unit': 'MP/s',
        'n_gpus': world, 'steps': args.steps, 'warmup': warmup, 'ms_per_step': sub['ms_per_step'],
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f16',
        'data': 'synthetic',
        'config': {'workload': f'{ARCH_TEXT.get(args.arch, args.arch)}, ' + sub['workload'],
                   'l2': 'flushed between timed iterations (256 MiB write, then read back)',
                   'accumulate': 'f32', 'est_bpp': sub['est_bpp']},
        'clocks': clk.summary(),
        'e2e': {'value': round(e2e_value, 2), 'unit': 'MP/s', 'h2d_bytes_per_step': int(x_pin.numel()),
                'd2h_bytes_per_step': int(x_pin.numel()) + 8},
        'gpu_launches': int((sub['launches_per_step'] or 0) * args.steps),
        'pipeline_tflops': sub['tflops'],
        'pipeline_tensor_frac': round(sub['tflops'] / peaks['bf16'], 4),
        'roofline': roof, 'cpu_baseline': None,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=8)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='wsi', choices=['wsi', 'patches', 'train'])
    ap.add_argument('--arch', default=ARCH_NAME)
    ap.add_argument('--batch', type=int, default=BATCH, help='patches per step (workload patches)')
    ap.add_argument('--tiles', type=int, default=TILES, help='512x512 chunks per GPU per step (workload wsi)')
    ap.add_argument('--batch-tiles', type=int, default=32, help='chunks per CUDA-graph replay')
    ap.add_argument('--coder-tiles', type=int, default=0,
                    help='chunk streams entropy-coded per device call of the device-resident run (0 = the shard)')
    ap.add_argument('--e2e-coder-tiles', default='0',
                    help='the same for compress_image (0 = the default schedule; one size, or a comma-separated '
                         'schedule of group sizes: the chunk files of one group are written while the next '
                         'group is on the GPU, so the last group is the exposed one)')
    ap.add_argument('--e2e-decoder-tiles', default='0',
                    help='the same for decompress_image (0 = the coder schedule reversed: the first group is '
                         'the exposed one)')
    ap.add_argument('--e2e-in-flight', type=int, default=2, choices=[1, 2],
                    help='steps in flight in the e2e region: 2 = the compress_image call of step k + 1 runs '
                         'beside the decompress_image call of step k (jobs.SlideJobs); 1 = one call after the other')
    ap.add_argument('--parity-tiles', type=int, default=8)
    ap.add_argument('--no-parity', action='store_true')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-graph', action='store_true',
                    help='issue every kernel from Python instead of replaying CUDA graphs')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the outputs of the last timed step as DIR/<name>.npy (workload wsi)')
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != 'ours' or args.workload != 'wsi'):
        ap.error('--dump-outputs writes the outputs of --workload wsi with --impl ours')
    if any(k in os.environ for k in ('CUDA_INJECTION64_PATH', 'NV_COMPUTE_PROFILER_PERFWORKS_DIR',
                                     'NV_NSIGHT_INJECTION_PORT_BASE')) and not args.no_graph:
        # ncu --set full cannot replay the tensor-map kernels as graph nodes (profiles/README.md)
        print('bench.py: profiler detected, launching kernels eagerly (no CUDA graph)', file=sys.stderr)
        args.no_graph = True
        os.environ['CAE_SLIDE_NO_GRAPHS'] = '1'
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    if args.impl == 'reference':
        return run_reference(args, rank, world)
    if args.workload == 'patches':
        return run_patches(args)
    if args.workload == 'train':
        from tools import trainbench
        return trainbench.run(args)
    return run_wsi(args)


if __name__ == '__main__':
    main()
