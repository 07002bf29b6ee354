"""Pyramid levels written by ``compress_image(..., levels=K)`` on the 12 x 13-chunk slide at PS = 64
with 40 px and 24 px edge chunks (levels 1..6: every level has ragged edges and level 6 is one
12 x 13 px chunk), ``batch_tiles`` 16 so that batches span chunk rows: the level files compared
byte for byte against ``compress_image`` of the exact reduction of the source, through the engine
(page-locked and pageable source) and the general loop."""
import json
import os

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


def _tree(path):
    """relative path -> (bytes, mtime_ns) of every file under ``path``, and -> None of every
    directory (an empty one included)."""
    out = {}
    for root, dirs, files in os.walk(path):
        for d in dirs:
            out[os.path.relpath(os.path.join(root, d), path) + '/'] = None
        for f in files:
            p = os.path.join(root, f)
            out[os.path.relpath(p, path)] = (open(p, 'rb').read(), os.stat(p).st_mtime_ns)
    return out


def _files(d):
    return {f: open(os.path.join(d, f), 'rb').read() for f in sorted(os.listdir(d))}


def _slide(gy, gx, cut_y, cut_x):
    from oracle import cae_oracle as O
    s = np.concatenate([np.concatenate([O.synth_tissue_tile(i, j, ps=PS, seed=2) for j in range(gx)],
                                       axis=1) for i in range(gy)], axis=0)
    return np.ascontiguousarray(s[:gy * PS - cut_y, :gx * PS - cut_x])


def _reference(tmp, chk, slide, levels):
    """level -> files of compress_image of the level image (level 0: of the slide)."""
    from cnn_autoencoder_b200 import compress
    out = {}
    for k in range(levels + 1):
        p = str(tmp / ('ref%d.zarr' % k))
        compress.compress_image('CAE', chk, reduce_ref(slide, 2 ** k) if k else slide, p,
                                patch_size=PS, batch_tiles=16)
        out[k] = _files(os.path.join(p, '0', '0'))
    return out


@pytest.fixture(scope='module')
def case(tmp_path_factory):
    from oracle import cae_oracle as O
    chk = O.make_checkpoint(ARCH, seed=9)
    slide = _slide(12, 13, 24, 40)
    return chk, slide, _reference(tmp_path_factory.mktemp('levels_ref'), chk, slide, K)


def _check(path, ref, levels, stats=None):
    from cnn_autoencoder_b200.region import multiscales
    for k in range(levels + 1):
        got = _files(os.path.join(path, '0', str(k)))
        assert sorted(got) == sorted(ref[k]), k
        bad = [f for f in got if got[f] != ref[k][f]]
        assert not bad, (k, bad)
    with open(os.path.join(path, '0', '.zattrs')) as f:
        assert json.load(f)['multiscales'] == json.loads(json.dumps(multiscales(levels)))
    assert os.path.exists(os.path.join(path, '.zgroup')) and os.path.exists(os.path.join(path, '0', '.zgroup'))
    if stats is not None:
        assert stats['level_chunks'] == sum(len(ref[k]) - 1 for k in range(1, levels + 1))
        assert stats['level_bytes'] == sum(len(b) for k in range(1, levels + 1)
                                           for f, b in ref[k].items() if f != '.zarray')
        assert stats['bytes'] == sum(len(b) for f, b in ref[0].items() if f != '.zarray')


@pytest.mark.parametrize('route', ['engine_pinned', 'engine_pageable', 'general', 'device_coder'])
def test_levels_equal_compress_image_of_the_reduction(case, route, tmp_path, monkeypatch):
    from cnn_autoencoder_b200 import compress
    chk, slide, ref = case
    src = slide
    if route == 'engine_pinned':
        src = torch.from_numpy(slide).pin_memory().numpy()
    if route == 'general':
        monkeypatch.setenv('CAE_NO_SLIDE_ENGINE', '1')
    fe = compress.load_model(chk)['fact_ent'].module
    if route == 'device_coder':
        monkeypatch.setattr(fe, 'GPU_CODER_MIN_STREAMS', 16)     # the level groups too (62 tiles)
    path = str(tmp_path / 'slide.zarr')
    st = compress.compress_image('CAE', chk, src, path, patch_size=PS, batch_tiles=16, levels=K)
    assert st['tiles'] == 156 and st['pixels'] == 156 * PS * PS
    assert (st.get('engine') == 'slide') == (route != 'general')
    assert st['level_chunks'] == LEVEL_TILES
    _check(path, ref, K, st)


def test_small_slide_general_loop_and_auto(tmp_path):
    """Under 128 chunks the general loop runs by itself; 'auto' is default_levels."""
    from oracle import cae_oracle as O
    from cnn_autoencoder_b200 import compress
    from cnn_autoencoder_b200.region import default_levels
    chk = O.make_checkpoint(ARCH, seed=5)
    slide = _slide(7, 9, 20, 0)
    K_auto = default_levels(slide.shape, PS)
    assert K_auto == 4
    ref = _reference(tmp_path, chk, slide, K_auto)
    path = str(tmp_path / 'small.zarr')
    st = compress.compress_image('CAE', chk, slide, path, patch_size=PS, batch_tiles=16,
                                 levels='auto')
    assert 'engine' not in st
    _check(path, ref, K_auto, st)
    assert not os.path.exists(os.path.join(path, '0', str(K_auto + 1)))


def test_no_levels_is_unchanged_and_levels_read_back(case, tmp_path):
    from cnn_autoencoder_b200 import compress, decompress
    from cnn_autoencoder_b200.region import CompressedSlide
    chk, slide, ref = case
    path = str(tmp_path / 'plain.zarr')
    st = compress.compress_image('CAE', chk, slide, path, patch_size=PS, batch_tiles=16)
    assert 'level_chunks' not in st and sorted(os.listdir(path)) == ['0']
    assert sorted(os.listdir(os.path.join(path, '0'))) == ['0']
    assert _files(os.path.join(path, '0', '0')) == ref[0]
    path = str(tmp_path / 'levels.zarr')
    compress.compress_image('CAE', chk, slide, path, patch_size=PS, batch_tiles=16, levels=K)
    with CompressedSlide(path, chk, batch_tiles=16) as s:
        assert s.levels == list(range(K + 1))
        for k in (1, 3, 6):
            lv = s.level(k)
            whole = torch.zeros(lv.shape, dtype=torch.uint8).pin_memory().numpy()
            decompress.decompress_image(path, whole, data_group='0/%d' % k, checkpoint=chk,
                                        batch_tiles=16)
            assert np.array_equal(lv[:], whole), k
            ly, lx, _ = lv.shape
            h, w = max(1, ly // 2), max(1, lx // 3)
            assert np.array_equal(lv.read_region(ly - h, lx - w, h, w).cpu().numpy(),
                                  whole[ly - h:, lx - w:])


def test_overwrite_over_a_built_pyramid(case, tmp_path):
    from cnn_autoencoder_b200 import compress
    from cnn_autoencoder_b200.region import CompressedSlide, stored_levels
    chk, slide, ref = case
    path = str(tmp_path / 'over.zarr')
    compress.compress_image('CAE', chk, slide[::-1].copy(), path, patch_size=PS, batch_tiles=16)
    with open(os.path.join(path, '0', '.zattrs'), 'w') as f:
        json.dump({'note': 'kept'}, f)
    with CompressedSlide(path, chk, mode='r+', batch_tiles=16) as s:
        s.build_pyramid(levels=K)
    upper = {k: _tree(os.path.join(path, '0', str(k))) for k in range(4, K + 1)}
    st = compress.compress_image('CAE', chk, slide, path, patch_size=PS, batch_tiles=16, levels=3)
    assert st['level_chunks'] == 6 * 7 + 3 * 4 + 2 * 2
    _check(path, ref, 3, st)
    assert stored_levels(os.path.join(path, '0')) == [0, 1, 2, 3]
    with open(os.path.join(path, '0', '.zattrs')) as f:
        assert json.load(f)['note'] == 'kept'
    for k in range(4, K + 1):
        assert _tree(os.path.join(path, '0', str(k))) == upper[k], k        # bytes and mtimes
    with CompressedSlide(path, chk, mode='r+', batch_tiles=16) as s:
        assert s.levels == [0, 1, 2, 3]
        s.build_pyramid(levels=K, overwrite=True)
        assert s.levels == list(range(K + 1))


def test_refusals_touch_nothing(case, tmp_path):
    from cnn_autoencoder_b200 import compress
    chk, slide, _ = case
    path = str(tmp_path / 'store.zarr')
    compress.compress_image('CAE', chk, slide, path, patch_size=PS, batch_tiles=16, levels=2)
    before = _tree(str(tmp_path))
    for kw in (dict(levels=3, save_as_bottleneck=True), dict(levels='auto', world_size=2, rank=0),
               dict(levels=2, data_group='0/1'), dict(levels=7), dict(levels=True),
               dict(levels=-1)):
        for out in (path, str(tmp_path / 'new.zarr')):
            with pytest.raises(ValueError):
                compress.compress_image('CAE', chk, slide, out, patch_size=PS, batch_tiles=16, **kw)
    assert _tree(str(tmp_path)) == before
    assert not os.path.exists(str(tmp_path / 'new.zarr'))


def test_engine_refuses_levels_with_a_device_source(case):
    from cnn_autoencoder_b200 import _slide, compress
    chk, slide, _ = case
    tc = _slide.tile_codec(compress.load_model(chk), PS, 3, 16)
    x = torch.zeros((4, PS, PS, 3), dtype=torch.uint8, device='cuda')
    with pytest.raises(ValueError, match='device_source'):
        _slide.compress_tiles(tc, None, [(0, j) for j in range(4)], lambda idx: 'unused', (PS, PS),
                              2, 16, _slide._Stats(), device_source=x, level_arrays=[object()])


def test_beside_a_decompress_in_slide_jobs(case, tmp_path):
    """A compress with levels in flight beside a decompress gives the files of the calls one
    after the other."""
    from cnn_autoencoder_b200 import compress, decompress
    from cnn_autoencoder_b200.jobs import SlideJobs
    chk, slide, ref = case
    other = str(tmp_path / 'other.zarr')
    compress.compress_image('CAE', chk, slide[:, ::-1].copy(), other, patch_size=PS, batch_tiles=16)
    alone = torch.zeros(slide.shape, dtype=torch.uint8).pin_memory().numpy()
    decompress.decompress_image(other, alone, checkpoint=chk, batch_tiles=16)
    canvas = torch.zeros(slide.shape, dtype=torch.uint8).pin_memory().numpy()
    src = torch.from_numpy(slide).pin_memory().numpy()
    with SlideJobs() as jobs:
        for r in range(2):
            path = str(tmp_path / ('jobs%d.zarr' % r))
            a = jobs.submit('compress', compress.compress_image, 'CAE', chk, src, path,
                            patch_size=PS, batch_tiles=16, levels=K)
            b = jobs.submit('decompress', decompress.decompress_image, other, canvas,
                            checkpoint=chk, batch_tiles=16)
            st = a.result()
            b.result()
            _check(path, ref, K, st)
            assert np.array_equal(canvas, alone)
