"""Resolution pyramid geometry (``region.default_levels``, ``pyramid_rows``, ``pyramid_place``), its
metadata (``multiscales``, ``write_multiscales``, ``stored_levels``) and the host-side checks of
``cae_tiles_pyramid_u8``: no device."""
import ctypes
import json
import os

import numpy as np
import pytest

from cnn_autoencoder_b200 import _cabi as C
from cnn_autoencoder_b200.region import (check_levels, default_levels, level_shape, pyramid_place,
                                         pyramid_rows, stored_levels, write_multiscales)

SHAPES = [(12 * 64 - 24, 13 * 64 - 40, 64), (64, 64, 64), (1, 200, 16), (130, 1, 32),
          (300, 257, 32), (96, 80, 48)]


def _levels_up_to(ps):
    K = 0
    while ps % 2 ** (K + 1) == 0:
        K += 1
    return K


@pytest.mark.parametrize('Y, X, ps', SHAPES)
def test_level0_chunks_map_to_their_level_tiles(Y, X, ps):
    """Every in-array level-0 pixel of chunk (i, j) reduces into level pixel (y >> k, x >> k):
    the level chunk, the offset in it and the extent covered must be what pyramid_place says."""
    gy, gx = -(-Y // ps), -(-X // ps)
    chunk_yx = np.array([(i, j) for i in range(gy) for j in range(gx)])
    for k in range(1, _levels_up_to(ps) + 1):
        place = pyramid_place((Y, X, 3), ps, k, chunk_yx)
        ly, lx = level_shape((Y, X, 3), 2 ** k)[:2]
        cover = np.zeros((ly, lx), dtype=np.int64)
        for (i, j), (tile, oy, ox, eh, ew) in zip(chunk_yx, place):
            ys = np.arange(i * ps, min((i + 1) * ps, Y)) >> k         # level rows / columns hit
            xs = np.arange(j * ps, min((j + 1) * ps, X)) >> k
            ys, xs = np.unique(ys), np.unique(xs)
            assert set(ys // ps) == {i >> k} and set(xs // ps) == {tile}
            assert (ys.min() % ps, xs.min() % ps) == (oy, ox)
            assert (len(ys), len(xs)) == (eh, ew)
            assert ys.max() - ys.min() + 1 == eh and xs.max() - xs.min() + 1 == ew
            cover[np.ix_(ys, xs)] += 1
        assert (cover == 1).all()          # the chunks tile the level, no level pixel twice


@pytest.mark.parametrize('Y, X, ps', SHAPES)
def test_level_rows_complete_after_their_last_level0_row(Y, X, ps):
    gy = -(-Y // ps)
    K = _levels_up_to(ps)
    order = pyramid_rows(gy, K)
    assert len(order) == len(set(order))
    for k in range(1, K + 1):
        gk = -(-level_shape((Y, X, 3), 2 ** k)[0] // ps)
        assert sorted(R for kk, R in order if kk == k) == list(range(gk))
    # (k, R) comes after every level row whose last level-0 row precedes its own
    last = {(k, R): min(2 ** k * (R + 1), gy) - 1 for k, R in order}
    assert [last[o] for o in order] == sorted(last[o] for o in order)


@pytest.mark.parametrize('Y, X, ps', SHAPES + [(65536, 32768, 512), (512, 513, 512),
                                                (10 ** 6, 10, 512)])
def test_default_levels(Y, X, ps):
    cap = _levels_up_to(ps)
    fits = [K for K in range(1, cap + 1) if max(level_shape((Y, X, 3), 2 ** K)[:2]) <= ps]
    assert default_levels((Y, X, 3), ps) == (fits[0] if fits else cap)
    assert default_levels((65536, 32768, 3), 512) == 7


@pytest.mark.parametrize('K, ps', [(0, 64), (-1, 64), (7, 64), (5, 48), (1, 15), (True, 64),
                                   (2.0, 64)])
def test_bad_level_counts_are_refused(K, ps):
    with pytest.raises(ValueError):
        check_levels(K, ps)


def test_multiscales_metadata(tmp_path):
    store = str(tmp_path / 's.zarr')
    group = os.path.join(store, '0')
    os.makedirs(os.path.join(group, '0'))
    with open(os.path.join(group, '.zattrs'), 'w') as f:
        json.dump({'omero': {'name': 'x'}, 'multiscales': [{'datasets': [{'path': '0'}]}]}, f)
    assert stored_levels(group) == [0]
    write_multiscales(store, group, 3)
    for d in (store, group):
        with open(os.path.join(d, '.zgroup')) as f:
            assert json.load(f) == {'zarr_format': 2}
    with open(os.path.join(group, '.zattrs')) as f:
        attrs = json.load(f)
    assert attrs['omero'] == {'name': 'x'}
    (ms,) = attrs['multiscales']
    assert ms['version'] == '0.4' and ms['type'] == 'mean'
    assert [a['name'] for a in ms['axes']] == ['y', 'x', 'c']
    assert [a['type'] for a in ms['axes']] == ['space', 'space', 'channel']
    assert [d['path'] for d in ms['datasets']] == ['0', '1', '2', '3']
    for k, d in enumerate(ms['datasets']):
        assert d['coordinateTransformations'] == [{'type': 'scale', 'scale': [2 ** k, 2 ** k, 1]}]
    assert stored_levels(group) == [0, 1, 2, 3]
    assert not [n for n in os.listdir(group) if n.endswith('.tmp')]
    write_multiscales(store, group, 0)                  # the entry goes, the other keys stay
    with open(os.path.join(group, '.zattrs')) as f:
        assert json.load(f) == {'omero': {'name': 'x'}}
    assert stored_levels(group) == [0]
    assert stored_levels(str(tmp_path / 'nothing')) == [0]


# ---- host-side checks of cae_tiles_pyramid_u8 (fake device pointers: never dereferenced) ----
_FAKE = ctypes.c_void_p(1 << 20)
GOOD = [1, 2, 16, 16]


def _pyramid(recs, ps=16, c=3, levels=2, gy=3, gx=4, tiles=_FAKE, recs_dev=_FAKE, out=_FAKE,
             n_tiles=None):
    r = np.ascontiguousarray(recs, dtype=np.int32).reshape(-1, 4)
    rc = C.lib().cae_tiles_pyramid_u8(tiles, len(r) if n_tiles is None else n_tiles, ps, c, levels,
                                      r.ctypes.data if len(r) else None, recs_dev, gy, gx, out,
                                      None)
    return rc, C.lib().cae_last_error().decode()


@pytest.mark.parametrize('levels, ps', [(0, 16), (-1, 16), (5, 16), (10, 1024), (2, 6), (1, 9)])
def test_pyramid_refuses_a_bad_level_count(levels, ps):
    rc, msg = _pyramid([GOOD, [9, 9, 9, 9]], ps=ps, levels=levels)
    assert rc == 2 and 'cae_tiles_pyramid_u8' in msg and '%d levels' % levels in msg, msg


@pytest.mark.parametrize('bad, what', [
    ([3, 0, 16, 16], 'chunk (3, 0) of a 3 x 4 grid'),
    ([-1, 0, 16, 16], 'chunk (-1, 0)'),
    ([0, 4, 16, 16], 'chunk (0, 4)'),
    ([0, -1, 16, 16], 'chunk (0, -1)'),
    ([0, 0, 0, 16], 'in-array extent 0 x 16'),
    ([0, 0, 16, 17], 'in-array extent 16 x 17'),
    ([0, 0, 17, 1], 'in-array extent 17 x 1'),
    ([0, 0, 5, -3], 'in-array extent 5 x -3'),
    ([2, 0, 16, 16], 'different level-1 chunk rows'),            # record 0 is in row 1
])
def test_pyramid_refuses_a_bad_record(bad, what):
    rc, msg = _pyramid([GOOD, bad])
    assert rc == 2 and 'cae_tiles_pyramid_u8' in msg and 'record 1' in msg and what in msg, msg


def test_pyramid_accepts_ragged_extents():
    # a 1 x 1 edge chunk passes; the call then fails on the next record, which proves it did
    rc, msg = _pyramid([[1, 3, 1, 1], [0, 0, 16, 0]])
    assert rc == 2 and 'record 1' in msg, msg


def test_pyramid_refuses_null_pointers_misalignment_and_bad_arguments():
    for kw in (dict(tiles=None), dict(recs_dev=None), dict(out=None)):
        rc, msg = _pyramid([GOOD], **kw)
        assert rc == 2 and 'null pointer' in msg, (kw, msg)
    rc, msg = _pyramid([], n_tiles=1)
    assert rc == 2 and 'null pointer' in msg, msg
    rc, msg = _pyramid([GOOD], recs_dev=ctypes.c_void_p((1 << 20) + 4))
    assert rc == 2 and 'aligned' in msg, msg
    for kw in (dict(ps=0), dict(c=0), dict(gy=0), dict(gx=-1), dict(n_tiles=-1),
               dict(n_tiles=70000)):
        rc, msg = _pyramid([GOOD], **kw)
        assert rc == 2 and 'bad argument' in msg, (kw, msg)
    rc, msg = _pyramid([GOOD], ps=512, levels=9, c=16)
    assert rc == 2 and 'shared memory' in msg, msg
    assert _pyramid([], n_tiles=0)[0] == 0                  # nothing to do, nothing touched
