"""Region writes (``region.CompressedSlide`` in mode 'r+', ``create_slide``, ``cae_tiles_paste_u8``)
on a 12 x 13-chunk slide at PS = 64 with 40 px and 24 px edge chunks: chunk files compared byte
for byte against ``compress_image`` and against the codec class's read-modify-write."""
import ctypes
import os
import shutil
import struct

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ARCH = dict(channels_org=3, channels_net=32, channels_bn=16, compression_level=3,
            act_layer_type='LeakyReLU')
PS = 64


def _slide(gy, gx, crop):
    from oracle import cae_oracle as O
    s = np.concatenate([np.concatenate([O.synth_tissue_tile(i, j, ps=PS, seed=2) for j in range(gx)],
                                       axis=1) for i in range(gy)], axis=0)
    return np.ascontiguousarray(s[:s.shape[0] - crop[0], :s.shape[1] - crop[1]])


def _pinned(shape):
    return torch.zeros(shape, dtype=torch.uint8).pin_memory().numpy()


@pytest.fixture(scope='module')
def store(tmp_path_factory):
    """(store path written by compress_image, checkpoint, the source slide)."""
    from oracle import cae_oracle as O
    from cnn_autoencoder_b200 import compress
    chk = O.make_checkpoint(ARCH, seed=9)
    slide = _slide(12, 13, (24, 40))
    path = str(tmp_path_factory.mktemp('region_write') / 'slide.zarr')
    compress.compress_image('CAE', chk, slide, path, patch_size=PS, batch_tiles=16, coder_tiles=96)
    return path, chk, slide


@pytest.fixture
def copy(store, tmp_path):
    """A fresh copy of the store for one test."""
    dst = str(tmp_path / 'copy.zarr')
    shutil.copytree(store[0], dst)
    return dst


@pytest.fixture(scope='module')
def codec(store):
    from cnn_autoencoder_b200._autoencoders import ConvolutionalAutoencoder
    return ConvolutionalAutoencoder(store[1])


def _arr_dir(path):
    return os.path.join(path, '0/0')


def _files(path):
    """name -> (bytes, inode) of every chunk file."""
    d = _arr_dir(path)
    return {f: (open(os.path.join(d, f), 'rb').read(), os.stat(os.path.join(d, f)).st_ino)
            for f in sorted(os.listdir(d)) if not f.startswith('.')}


def _touched(y, x, h, w):
    return {(iy, ix) for iy in range(y // PS, (y + h - 1) // PS + 1)
            for ix in range(x // PS, (x + w - 1) // PS + 1)}


def _rmw(codec, old_bytes, iy, ix, value, y, x, H, W):
    """The codec class's read-modify-write of chunk (iy, ix): decode the old file (or zeros),
    paste the window ``value`` at (y, x), zero the part beyond the array edge, encode."""
    tile = codec.decode(old_bytes).copy() if old_bytes is not None else np.zeros((PS, PS, 3), np.uint8)
    h, w = value.shape[:2]
    a, b = max(y, iy * PS), min(y + h, (iy + 1) * PS)
    c, d = max(x, ix * PS), min(x + w, (ix + 1) * PS)
    tile[a - iy * PS:b - iy * PS, c - ix * PS:d - ix * PS] = value[a - y:b - y, c - x:d - x]
    tile[max(0, H - iy * PS):] = 0
    tile[:, max(0, W - ix * PS):] = 0
    return codec.encode(tile)


def test_chunk_aligned_writes_equal_compress_image(store, tmp_path):
    from cnn_autoencoder_b200.region import create_slide
    path, chk, slide = store
    H, W, _ = slide.shape
    want = _files(path)
    meta = open(os.path.join(_arr_dir(path), '.zarray')).read()
    strips = str(tmp_path / 'strips.zarr')
    with create_slide(strips, chk, slide.shape, patch_size=PS) as s:
        assert s.mode == 'r+' and s.shape == slide.shape
        assert not s[:, :].any()                                     # no chunk yet: all fill value
        for y0 in range(0, H, 2 * PS):                               # 2 chunk rows; the last ragged
            s[y0:y0 + 2 * PS] = slide[y0:y0 + 2 * PS]
            assert s.stats['full'] == s.stats['chunks'] == s.stats['missing'] == 2 * 13
            assert s.stats['decoded'] == s.stats['partial'] == 0
    whole = str(tmp_path / 'whole.zarr')
    with create_slide(whole, chk, slide.shape, patch_size=PS) as s:
        s[:, :] = slide
        assert s.stats['device_coded'] == s.stats['chunks'] == 156
    for out in (strips, whole):
        assert open(os.path.join(_arr_dir(out), '.zarray')).read() == meta
        got = _files(out)
        assert sorted(got) == sorted(want)
        bad = [f for f in want if got[f][0] != want[f][0]]
        assert not bad, (out, bad)


def test_partial_writes_follow_zarr_read_modify_write(store, copy, codec):
    from cnn_autoencoder_b200 import decompress
    from cnn_autoencoder_b200.region import CompressedSlide
    _, chk, slide = store
    H, W, _ = slide.shape
    rng = np.random.default_rng(21)
    writes = [(10, 5, 40, 50),                          # inside one chunk
              (3 * PS - 20, 5 * PS - 30, 50, 70),       # across a 2 x 2 chunk corner
              (H - 30, W - 50, 30, 50),                 # the ragged bottom-right edge
              (100, 200, 80, 60)]                       # a scalar redaction
    with CompressedSlide(copy, chk, mode='r+') as s:
        for n, (y, x, h, w) in enumerate(writes):
            before = _files(copy)
            if n < 3:
                value = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
                s[y:y + h, x:x + w] = value
            else:
                value = np.zeros((h, w, 3), dtype=np.uint8)
                s[y:y + h, x:x + w] = 0
            touched = _touched(y, x, h, w)
            assert s.stats['chunks'] == s.stats['decoded'] == s.stats['partial'] == len(touched)
            after = _files(copy)
            assert sorted(after) == sorted(before)
            for f in before:
                iy, ix, _ = map(int, f.split('.'))
                if (iy, ix) in touched:
                    want = _rmw(codec, before[f][0], iy, ix, value, y, x, H, W)
                    assert after[f][0] == want, (n, f)
                else:
                    assert after[f] == before[f], (n, f)            # same bytes, same inode
        got = s[:, :]
    canvas = _pinned(slide.shape)
    decompress.decompress_image(copy, canvas, checkpoint=chk, batch_tiles=16, coder_tiles=96)
    assert np.array_equal(got, canvas)


def test_input_forms_and_coders_give_the_same_files(store, tmp_path):
    from cnn_autoencoder_b200.region import CompressedSlide
    path, chk, slide = store
    H, W, _ = slide.shape
    rng = np.random.default_rng(4)
    h, w = 70, 90
    boxes = []                                  # non-overlapping boxes by rejection sampling
    taken = np.zeros((H, W), dtype=bool)
    while len(boxes) < 12:
        y, x = int(rng.integers(0, H - h + 1)), int(rng.integers(0, W - w + 1))
        if not taken[y:y + h, x:x + w].any():
            taken[y:y + h, x:x + w] = True
            boxes.append((y, x))
    vals = rng.integers(0, 256, size=(len(boxes), h, w, 3), dtype=np.uint8)
    pinned = _pinned(vals.shape)
    pinned[:] = vals
    results = {}
    forms = [('cuda', torch.from_numpy(vals).cuda(), None), ('pinned', pinned, None),
             ('host', vals.copy(), None), ('device_coder', vals, 1), ('host_coder', vals, 10 ** 9)]
    for name, v, threshold in forms:
        out = str(tmp_path / (name + '.zarr'))
        shutil.copytree(path, out)
        with CompressedSlide(out, chk, mode='r+', batch_tiles=8) as s:
            if threshold is not None:
                s.fact_ent.GPU_CODER_MIN_STREAMS = threshold        # instance override, this reader only
            s.write_regions(boxes, h, w, v)
            st = s.stats
            if name == 'device_coder':
                assert st['device_coded'] == st['chunks'] and st['device_decoded'] == st['decoded'] > 0
            if name == 'host_coder':
                assert st['device_coded'] == st['device_decoded'] == 0
        results[name] = _files(out)
    ref = results['cuda']
    for name in results:
        assert {f: b for f, (b, _) in results[name].items()} == {f: b for f, (b, _) in ref.items()}, name
    for f, (b_, _) in ref.items():                       # untouched chunks keep their bytes
        iy, ix, _ = map(int, f.split('.'))
        if not any((iy, ix) in _touched(by, bx, h, w) for by, bx in boxes):
            assert b_ == _files(path)[f][0], f
    # one window through __setitem__ and write_region; a colour broadcast and spelled out
    y, x = boxes[0]
    colour = np.array([200, 30, 90], dtype=np.uint8)
    writes = {'setitem': lambda s: s.__setitem__((slice(y, y + h), slice(x, x + w)), vals[0]),
              'write_region': lambda s: s.write_region(y, x, torch.from_numpy(vals[0]).cuda()),
              'colour': lambda s: s.__setitem__((slice(y, y + h), slice(x, x + w)), colour),
              'colour_array': lambda s: s.__setitem__((slice(y, y + h), slice(x, x + w)),
                                                      np.ascontiguousarray(np.broadcast_to(colour, (h, w, 3))))}
    got = {}
    for name, fn in writes.items():
        out = str(tmp_path / (name + '.zarr'))
        shutil.copytree(path, out)
        with CompressedSlide(out, chk, mode='r+') as s:
            fn(s)
            assert s.stats['chunks'] == len(_touched(y, x, h, w))
            if name == 'colour':
                s[5, 10:20] = colour                                          # a row: (3,) broadcast
                assert s.stats['chunks'] == 1
                s[5:7, 3] = np.array([[1, 2, 3], [4, 5, 6]], dtype=np.uint8)  # a column
                assert s.stats['chunks'] == 1
                s[10:10, :] = 7                                               # empty: a no-op
                assert s.stats['chunks'] == 1
        got[name] = {f: b_ for f, (b_, _) in _files(out).items()}
    assert got['setitem'] == got['write_region']
    colour_chunks = {'%d.%d.0' % t for t in _touched(y, x, h, w)}
    assert all(got['colour'][f] == got['colour_array'][f] for f in colour_chunks)


def test_missing_chunks(store, copy, codec):
    from cnn_autoencoder_b200.region import CompressedSlide
    _, chk, slide = store
    H, W, _ = slide.shape
    d = _arr_dir(copy)
    os.remove(os.path.join(d, '4.5.0'))
    os.remove(os.path.join(d, '11.12.0'))                # the ragged bottom-right corner chunk
    rng = np.random.default_rng(8)
    with CompressedSlide(copy, chk, mode='r+') as s:
        y, x = 4 * PS + 10, 5 * PS + 7                    # partly covers the missing chunk (4, 5)
        v = rng.integers(0, 256, size=(20, 30, 3), dtype=np.uint8)
        s[y:y + 20, x:x + 30] = v
        assert s.stats['missing'] == 1 and s.stats['decoded'] == 0 and s.stats['partial'] == 1
        want = _rmw(codec, None, 4, 5, v, y, x, H, W)
        assert open(os.path.join(d, '4.5.0'), 'rb').read() == want
        y, x = 11 * PS, 12 * PS                           # covers the missing edge chunk whole
        v = rng.integers(0, 256, size=(H - y, W - x, 3), dtype=np.uint8)
        s[y:, x:] = v
        assert s.stats['missing'] == s.stats['full'] == 1 and s.stats['decoded'] == 0
        tile = np.zeros((PS, PS, 3), dtype=np.uint8)
        tile[:H - y, :W - x] = v
        assert open(os.path.join(d, '11.12.0'), 'rb').read() == codec.encode(tile)


def test_refusals_touch_no_file(store, copy, tmp_path):
    from oracle import cae_oracle as O
    from cnn_autoencoder_b200 import _cabi as C, compress
    from cnn_autoencoder_b200.region import CompressedSlide, create_slide
    _, chk, slide = store

    def snapshot():
        d = _arr_dir(copy)
        return {f: (open(os.path.join(d, f), 'rb').read(), os.stat(os.path.join(d, f)).st_ino,
                    os.stat(os.path.join(d, f)).st_mtime_ns) for f in sorted(os.listdir(d))}
    before = snapshot()
    with CompressedSlide(copy, chk) as r:
        with pytest.raises(ValueError, match="mode='r\\+'"):
            r[0:10, 0:10] = 0
        with pytest.raises(ValueError, match="mode='r\\+'"):
            r.write_regions([(0, 0)], 4, 4, np.zeros((1, 4, 4, 3), np.uint8))
    with CompressedSlide(copy, chk, mode='r+') as s:
        for value in (np.zeros((10, 11, 3), np.uint8), np.zeros((10, 10, 3), np.float32),
                      np.zeros((10, 10, 4), np.uint8), 256, -1,
                      torch.zeros((10, 10, 3), dtype=torch.int32, device='cuda'),
                      torch.zeros((10, 11, 3), dtype=torch.uint8, device='cuda')):
            with pytest.raises(ValueError):
                s[0:10, 0:10] = value
        with pytest.raises(TypeError):
            s[0:10, 0:10] = 1.5
        with pytest.raises(ValueError):
            s.write_regions([(0, 0)], 10, 10, np.zeros((1, 10, 10, 3), np.int16))
        with pytest.raises(ValueError, match='overlap'):
            s.write_regions([(0, 0), (100, 100), (5, 5)], 10, 10, np.zeros((3, 10, 10, 3), np.uint8))
        with pytest.raises(ValueError):
            s.write_region(slide.shape[0] - 5, 0, np.zeros((10, 10, 3), np.uint8))
        assert snapshot() == before
        with pytest.raises(FileExistsError):
            create_slide(copy, chk, slide.shape, patch_size=PS)
        assert snapshot() == before
        # an old chunk whose header is not (ps, ps): the write raises, the file stays as it was
        f = os.path.join(_arr_dir(copy), '2.3.0')
        raw = open(f, 'rb').read()
        with open(f, 'wb') as fh:
            fh.write(struct.pack('>QQ', PS, PS // 2) + raw[16:])
        before = snapshot()
        with pytest.raises(C.CaeError, match='header'):
            s[2 * PS + 5:2 * PS + 15, 3 * PS + 5:3 * PS + 15] = 9
        assert snapshot() == before
    # 'cae_bn' stores are refused for writing as for reading
    chk_bn = O.make_checkpoint(ARCH, seed=17)
    lat = str(tmp_path / 'lat.zarr')
    compress.compress_image('CAE', chk_bn, np.ascontiguousarray(slide[:192, :256]), lat, patch_size=64,
                            save_as_bottleneck=True, batch_tiles=4)
    files = sorted(os.listdir(_arr_dir(lat)))
    with pytest.raises(ValueError, match='decompress_image'):
        CompressedSlide(lat, chk_bn, mode='r+')
    assert sorted(os.listdir(_arr_dir(lat))) == files


def _paste_case(c, mode, rng):
    """Boxes, pieces (quadrants of the top 44 rows of every tile; one fill piece) and the
    numpy result; rows 44.. of every tile are never written."""
    n_tiles, ps, n_boxes = 4, 64, 3
    bh, bw = (48, 64) if mode != 'unaligned' else (48, 61)
    quads = ((0, 32), (32, 32)) if mode != 'unaligned' else ((3, 29), (32, 27))
    boxes = rng.integers(0, 256, size=(n_boxes, bh, bw, c), dtype=np.uint8)
    want = np.full((n_tiles, ps, ps, c), 77, dtype=np.uint8)
    pieces = []
    for k in range(n_tiles):
        for sy, h in ((0, 24), (24, 20)):
            for sx, w in quads:
                b = -1 if (k, sy, sx) == (2, 24, quads[1][0]) else int(rng.integers(0, n_boxes))
                dy = int(rng.integers(0, bh - h + 1))
                if mode == 'unaligned':
                    dx = int(rng.integers(0, bw - w + 1))
                else:
                    dx = 16 * int(rng.integers(0, (bw - w) // 16 + 1))
                pieces.append([k, b, sy, sx, dy, dx, h, w])
                want[k, sy:sy + h, sx:sx + w] = 0 if b < 0 else boxes[b, dy:dy + h, dx:dx + w]
    return boxes, np.array(pieces, dtype=np.int32), want


@pytest.mark.parametrize('mode', ['aligned', 'unaligned', 'aligned_box_offset'])
@pytest.mark.parametrize('c', [1, 3, 4])
def test_paste_kernel_equals_numpy(c, mode):
    from cnn_autoencoder_b200 import _cabi as C
    rng = np.random.default_rng(c * 10 + len(mode))
    boxes, pieces, want = _paste_case(c, mode, rng)
    shift = 4 if mode == 'aligned_box_offset' else 0          # a box base off the 16-byte grid
    bbuf = torch.zeros(boxes.size + shift, dtype=torch.uint8, device='cuda')
    b = bbuf[shift:]
    b.copy_(torch.from_numpy(boxes.reshape(-1)))
    guard = 64
    tbuf = torch.full((want.size + 2 * guard,), 77, dtype=torch.uint8, device='cuda')
    tiles = tbuf[guard:guard + want.size]
    pdev = torch.empty(pieces.size, dtype=torch.int32, device='cuda')
    C.check(C.lib().cae_tiles_paste_u8(tiles.data_ptr(), want.shape[0], want.shape[1], c,
                                       pieces.ctypes.data, len(pieces), pdev.data_ptr(), b.data_ptr(),
                                       boxes.shape[0], boxes.shape[1], boxes.shape[2],
                                       ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    got = tbuf.cpu().numpy()
    assert np.array_equal(got[guard:guard + want.size].reshape(want.shape), want)
    assert (got[:guard] == 77).all() and (got[guard + want.size:] == 77).all()
