"""Resolution pyramids (``CompressedSlide.build_pyramid``, ``level``, ``cae_tiles_pyramid_u8``) on a
12 x 13-chunk slide at PS = 64 with 40 px and 24 px edge chunks, levels 1..6, so every level has
ragged edges and level 6 is one 12 x 13 px chunk: level files compared byte for byte against
``compress_image`` of the numpy reduction of what ``decompress_image`` writes."""
import os
import shutil

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ARCH = dict(channels_org=3, channels_net=32, channels_bn=16, compression_level=3,
            act_layer_type='LeakyReLU')
PS = 64
K = 6
LEVEL_TILES = 6 * 7 + 3 * 4 + 2 * 2 + 1 + 1 + 1


def reduce_ref(img, f):
    """The level-``f`` image of ``img`` (Y x X x c uint8): block means over the pixels inside
    the array, rounded half up."""
    Y, X, c = img.shape
    ly, lx = -(-Y // f), -(-X // f)
    pad = np.zeros((ly * f, lx * f, c), dtype=np.int64)
    pad[:Y, :X] = img
    s = pad.reshape(ly, f, lx, f, c).sum(axis=(1, 3))
    n = (np.minimum(f, Y - f * np.arange(ly))[:, None] * np.minimum(f, X - f * np.arange(lx)))[..., None]
    return ((s + n // 2) // n).astype(np.uint8)


def _array_files(d):
    """name -> (bytes, mtime_ns) of every file of the array directory ``d``, ``.zarray`` included."""
    return {f: (open(os.path.join(d, f), 'rb').read(), os.stat(os.path.join(d, f)).st_mtime_ns)
            for f in sorted(os.listdir(d))}


def _tree(path):
    """relative path -> (bytes, mtime_ns) of every file under ``path``."""
    out = {}
    for root, _, files in os.walk(path):
        for f in files:
            p = os.path.join(root, f)
            out[os.path.relpath(p, path)] = (open(p, 'rb').read(), os.stat(p).st_mtime_ns)
    return out


def _bytes(files):
    return {f: b for f, (b, _) in files.items()}


@pytest.fixture(scope='module')
def store(tmp_path_factory):
    """(store path, checkpoint, decompress_image's reconstruction of the whole slide)."""
    from oracle import cae_oracle as O
    from cnn_autoencoder_b200 import compress, decompress
    chk = O.make_checkpoint(ARCH, seed=9)
    s = np.concatenate([np.concatenate([O.synth_tissue_tile(i, j, ps=PS, seed=2) for j in range(13)],
                                       axis=1) for i in range(12)], axis=0)
    slide = np.ascontiguousarray(s[:12 * PS - 24, :13 * PS - 40])
    path = str(tmp_path_factory.mktemp('pyramid') / 'slide.zarr')
    compress.compress_image('CAE', chk, slide, path, patch_size=PS, batch_tiles=16, coder_tiles=96)
    canvas = torch.zeros(slide.shape, dtype=torch.uint8).pin_memory().numpy()
    decompress.decompress_image(path, canvas, checkpoint=chk, batch_tiles=16, coder_tiles=96)
    assert np.unique(canvas).size > 16
    return path, chk, slide, canvas


def _reference(tmp, chk, canvas, name):
    """level -> files of compress_image of the level image of ``canvas``."""
    from cnn_autoencoder_b200 import compress
    out = {}
    for k in range(1, K + 1):
        p = str(tmp / ('%s_ref%d.zarr' % (name, k)))
        compress.compress_image('CAE', chk, reduce_ref(canvas, 2 ** k), p, patch_size=PS,
                                batch_tiles=16)
        out[k] = _bytes(_array_files(os.path.join(p, '0', '0')))
    return out


@pytest.fixture(scope='module')
def reference(store, tmp_path_factory):
    _, chk, _, canvas = store
    return _reference(tmp_path_factory.mktemp('pyramid_ref'), chk, canvas, 'full')


@pytest.fixture(scope='module')
def built(store, tmp_path_factory):
    """A copy of the store with levels 1..6 built by a reader in mode 'r+'."""
    from cnn_autoencoder_b200.region import CompressedSlide
    path, chk, _, _ = store
    out = str(tmp_path_factory.mktemp('pyramid_built') / 'slide.zarr')
    shutil.copytree(path, out)
    level0 = _tree(os.path.join(out, '0', '0'))
    with CompressedSlide(out, chk, mode='r+', batch_tiles=16) as s:
        assert s.levels == [0]
        s.build_pyramid(levels=K)
        stats = dict(s.stats)
        assert s.levels == list(range(K + 1))
    assert _tree(os.path.join(out, '0', '0')) == level0          # bytes and mtimes
    return out, stats


def _check_levels(path, reference):
    for k in range(1, K + 1):
        got = _bytes(_array_files(os.path.join(path, '0', str(k))))
        assert sorted(got) == sorted(reference[k]), k
        bad = [f for f in got if got[f] != reference[k][f]]
        assert not bad, (k, bad)


def test_levels_equal_compress_image_of_the_reduction(built, reference):
    path, stats = built
    _check_levels(path, reference)
    assert stats['decoded'] == stats['chunks'] == 156 and stats['missing'] == 0
    assert stats['level_chunks'] == LEVEL_TILES
    for k in range(1, K + 1):
        assert len(reference[k]) - 1 == -(-(-(-(12 * PS - 24) // 2 ** k)) // PS) * \
            -(-(-(-(13 * PS - 40) // 2 ** k)) // PS)


def test_missing_chunks_reduce_as_zeros(store, tmp_path):
    from cnn_autoencoder_b200.region import CompressedSlide
    path, chk, _, canvas = store
    out = str(tmp_path / 'holes.zarr')
    shutil.copytree(path, out)
    holes = [(0, 0), (3, 5), (3, 6), (7, 12), (11, 12), (11, 0), (6, 2)]    # edge chunks among them
    zeroed = canvas.copy()
    for i, j in holes:
        os.remove(os.path.join(out, '0', '0', '%d.%d.0' % (i, j)))
        zeroed[i * PS:(i + 1) * PS, j * PS:(j + 1) * PS] = 0
    with CompressedSlide(out, chk, mode='r+', batch_tiles=16) as s:
        s.build_pyramid(levels=K)
        assert s.stats['decoded'] == 156 - len(holes) and s.stats['missing'] == len(holes)
    _check_levels(out, _reference(tmp_path, chk, zeroed, 'holes'))


def test_device_and_host_coders_write_the_same_files(store, built, tmp_path):
    from cnn_autoencoder_b200.region import CompressedSlide
    path, chk, _, _ = store
    want = {k: _bytes(_array_files(os.path.join(built[0], '0', str(k)))) for k in range(1, K + 1)}
    for name, threshold, coded in (('device', 1, LEVEL_TILES), ('host', 10 ** 9, 0)):
        out = str(tmp_path / (name + '.zarr'))
        shutil.copytree(path, out)
        with CompressedSlide(out, chk, mode='r+', batch_tiles=8) as s:
            s.fact_ent.GPU_CODER_MIN_STREAMS = threshold        # instance override, this reader only
            s.build_pyramid(levels=K)
            assert s.stats['device_coded'] == coded, name
        _check_levels(out, want)


@pytest.mark.parametrize('c, offset, ps, levels', [(3, 0, 64, 6), (1, 0, 64, 6), (3, 1, 64, 6),
                                                   (3, 0, 256, 8), (3, 0, 512, 7), (1, 1, 256, 3)])
def test_kernel_alone_on_ragged_tiles(c, offset, ps, levels):
    """Every level of random tiles against numpy; bytes outside the written parts keep a
    sentinel.  offset 1 misaligns the tiles (the byte-wise staging path); ps > 64 with levels
    above 6 folds the staged squares' totals."""
    from cnn_autoencoder_b200 import _cabi as C
    from cnn_autoencoder_b200.region import pyramid_place
    rng = np.random.default_rng(c + 10 * offset + ps + levels)
    gy, gx = 4, 5                                  # one call: chunks of one level-1 chunk row
    ij = [(2, 0), (3, 3), (3, 4), (2, 2), (2, 4), (3, 1), (3, 0)]
    vh = [ps, ps, 17, 33, ps, ps, 1]
    vw = [ps, ps, 1, ps, 40, ps, ps * 3 // 4]
    recs = np.array([[i, j, h, w] for (i, j), h, w in zip(ij, vh, vw)], dtype=np.int32)
    n = len(recs)
    tiles_h = rng.integers(0, 256, size=(n, ps, ps, c), dtype=np.uint8)
    raw = torch.empty(n * ps * ps * c + 16, dtype=torch.uint8, device='cuda')
    tiles = raw[offset:offset + n * ps * ps * c]
    tiles.copy_(torch.from_numpy(tiles_h.ravel()))
    widths = [-(-gx // 2 ** k) for k in range(1, levels + 1)]
    first = np.concatenate([[0], np.cumsum(widths)])
    out = torch.full((int(first[-1]), ps, ps, c), 77, dtype=torch.uint8, device='cuda')
    recs_dev = torch.empty(4 * n, dtype=torch.int32, device='cuda')
    stream = torch.cuda.current_stream().cuda_stream
    C.check(C.lib().cae_tiles_pyramid_u8(tiles.data_ptr(), n, ps, c, levels, recs.ctypes.data,
                                         recs_dev.data_ptr(), gy, gx, out.data_ptr(), stream))
    got = out.cpu().numpy()
    want = np.full_like(got, 77)
    for k in range(1, levels + 1):
        place = pyramid_place((gy * ps, gx * ps, c), ps, k, recs[:, :2])
        for t, (i, j, h, w) in enumerate(recs):
            tile, oy, ox = place[t][:3]
            lvl = reduce_ref(tiles_h[t, :h, :w], 2 ** k)
            want[first[k - 1] + tile, oy:oy + lvl.shape[0], ox:ox + lvl.shape[1]] = lvl
    for k in range(1, levels + 1):
        assert np.array_equal(got[first[k - 1]:first[k]], want[first[k - 1]:first[k]]), k


def test_level_reads_equal_the_stored_arrays(store, built):
    from cnn_autoencoder_b200 import decompress
    from cnn_autoencoder_b200.region import CompressedSlide, level_shape
    path, _ = built
    chk = store[1]
    with CompressedSlide(path, chk, batch_tiles=16) as s:
        assert s.levels == list(range(K + 1))
        assert s.level(0) is s
        with pytest.raises(KeyError):
            s.level(K + 1)
        for k in (1, 2, 4, 6):
            lv = s.level(k)
            assert lv.downsample == 2 ** k and lv.chunks == (PS, PS, 3)
            assert lv.shape == level_shape(s.shape, 2 ** k)
            ly, lx, _ = lv.shape
            whole = torch.zeros(lv.shape, dtype=torch.uint8).pin_memory().numpy()
            decompress.decompress_image(path, whole, data_group='0/%d' % k, checkpoint=chk,
                                        batch_tiles=16)
            with CompressedSlide(path, chk, data_group='0/%d' % k, batch_tiles=16) as fresh:
                assert fresh.levels == [0]
                h, w = max(1, min(50, ly // 2)), max(1, min(70, lx // 2))   # every box fits
                boxes = [(0, 0), (ly - h, lx - w), (ly // 3, lx // 4)]
                for y, x in boxes:
                    a = lv.read_region(y, x, h, w)
                    assert s.stats['decoded'] == s.stats['chunks']
                    assert np.array_equal(a.cpu().numpy(), fresh.read_region(y, x, h, w).cpu().numpy())
                    assert np.array_equal(a.cpu().numpy(), whole[y:y + h, x:x + w])
                batch = lv.read_regions(boxes, h, w)
                assert np.array_equal(batch.cpu().numpy(), np.stack([whole[y:y + h, x:x + w]
                                                                     for y, x in boxes]))
                host = np.empty((len(boxes), h, w, 3), dtype=np.uint8)
                assert lv.read_regions(boxes, h, w, out=host) is host
                assert np.array_equal(host, batch.cpu().numpy())
                dev = torch.empty((h, w, 3), dtype=torch.uint8, device='cuda')
                assert lv.read_region(*boxes[2], h, w, out=dev) is dev
                assert np.array_equal(dev.cpu().numpy(), whole[boxes[2][0]:boxes[2][0] + h,
                                                               boxes[2][1]:boxes[2][1] + w])
                assert np.array_equal(lv[:], whole) and np.array_equal(lv[3, 2:9], whole[3, 2:9])
            with pytest.raises(TypeError):
                lv[0:1, 0:1] = 0


def test_refusals_touch_nothing_and_overwrite_rebuilds(store, built, tmp_path):
    from cnn_autoencoder_b200.region import CompressedSlide
    path, chk, _, _ = store
    before = _tree(built[0])
    with CompressedSlide(built[0], chk, batch_tiles=16) as s:
        with pytest.raises(ValueError, match="mode='r\\+'"):
            s.build_pyramid()
    with CompressedSlide(built[0], chk, mode='r+', batch_tiles=16) as s:
        for bad in (0, 7, -1):
            with pytest.raises(ValueError):
                s.build_pyramid(levels=bad)
        with pytest.raises(FileExistsError):
            s.build_pyramid(levels=K)
        with pytest.raises(FileExistsError):
            s.build_pyramid()                                 # the default, 4, exists too
    with CompressedSlide(built[0], chk, data_group='0/2', mode='r+', batch_tiles=16) as s:
        with pytest.raises(ValueError, match='data group'):
            s.build_pyramid(levels=1)
    assert _tree(built[0]) == before
    # overwrite: a default build (K = 4) first, then all six levels again
    out = str(tmp_path / 'again.zarr')
    shutil.copytree(built[0], out)
    with CompressedSlide(out, chk, mode='r+', batch_tiles=16) as s:
        s.build_pyramid(overwrite=True)
        assert s.levels == [0, 1, 2, 3, 4]
        s.build_pyramid(levels=K, overwrite=True)
        assert s.levels == list(range(K + 1))
    assert _bytes(_tree(out)) == _bytes(before)


def test_create_slide_strips_give_the_same_levels(store, built, tmp_path):
    from cnn_autoencoder_b200.region import create_slide
    path, chk, slide, _ = store
    H = slide.shape[0]
    out = str(tmp_path / 'strips.zarr')
    with create_slide(out, chk, slide.shape, patch_size=PS) as s:
        for y0 in range(0, H, 2 * PS):
            s[y0:y0 + 2 * PS] = slide[y0:y0 + 2 * PS]
        s.build_pyramid(levels=K)
    for k in range(K + 1):
        assert _bytes(_array_files(os.path.join(out, '0', str(k)))) == \
            _bytes(_array_files(os.path.join(built[0], '0', str(k)))), k
