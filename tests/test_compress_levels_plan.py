"""Pyramid levels at compression time without a device: the argument checks of
``compress.check_levels``, the ``--levels`` flag, and the row-completion order of
``region.PyramidWriter`` (the helper shared with ``build_pyramid``) on ragged grids, with the
kernel launch replaced by a recorder."""
import numpy as np
import pytest
import torch

from cnn_autoencoder_b200 import _slide, compress
from cnn_autoencoder_b200.region import PyramidWriter, default_levels, pyramid_rows

SHAPE = (12 * 64 - 24, 13 * 64 - 40, 3)


def test_zero_and_auto():
    assert compress.check_levels(0, SHAPE, 64) == 0
    assert compress.check_levels(np.int64(0), SHAPE, 64) == 0
    assert compress.check_levels('auto', SHAPE, 64) == default_levels(SHAPE, 64) == 4
    assert compress.check_levels(6, SHAPE, 64) == 6
    # 0 is no pyramid whatever the other arguments say
    assert compress.check_levels(0, SHAPE, 64, save_as_bottleneck=True, world_size=4,
                                 data_group='0/2') == 0


@pytest.mark.parametrize('bad', [-1, 7, 30, True, False, 2.0, None, 'all', '3'])
def test_bad_levels(bad):
    with pytest.raises(ValueError):
        compress.check_levels(bad, SHAPE, 64)


@pytest.mark.parametrize('kw, match', [(dict(save_as_bottleneck=True), 'latent'),
                                       (dict(world_size=2), 'build_pyramid'),
                                       (dict(data_group='0/2'), 'data group'),
                                       (dict(data_group='0'), None),
                                       (dict(data_group=''), 'data group'),
                                       (dict(data_group='a/b/0/'), None)])
def test_refusals(kw, match):
    for levels in (3, 'auto'):
        if match is None:
            assert compress.check_levels(levels, SHAPE, 64, **kw) >= 1
        else:
            with pytest.raises(ValueError, match=match):
                compress.check_levels(levels, SHAPE, 64, **kw)


def test_cli_flag():
    base = ['-chk', 'm.pth', '-dd', 'a.npy', '-o', 'out.zarr']
    assert compress._parser().parse_args(base).levels == 0
    assert compress._parser().parse_args(base + ['--levels', '5']).levels == 5
    assert compress._parser().parse_args(base + ['--levels', 'auto']).levels == 'auto'
    with pytest.raises(SystemExit):
        compress._parser().parse_args(base + ['--levels', 'many'])


class _Recorder(PyramidWriter):
    """The writer with the kernel launch replaced: records which level rows were flushed when
    each level-0 chunk row segment was reduced."""

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        self.launches = []

    def _launch(self, tiles, a, b, ij):
        rows = set(ij[a:b, 0].tolist())
        assert len(rows) == 1
        self.launches.append((rows.pop(), list(self.flushed), b - a))


@pytest.mark.parametrize('Y, X, ps, K, batch', [(12 * 8 - 3, 13 * 8 - 5, 8, 3, 16),
                                                (12 * 8 - 3, 13 * 8 - 5, 8, 3, 5),
                                                (9 * 4, 3 * 4 - 1, 4, 2, 7),
                                                (1 * 8, 40 * 8, 8, 3, 16),
                                                (37 * 2, 1 * 2, 2, 1, 3),
                                                (17 * 8 - 1, 33 * 8 - 7, 8, 3, 13)])
def test_rows_complete_in_pyramid_rows_order(Y, X, ps, K, batch):
    gy, gx = -(-Y // ps), -(-X // ps)
    order = pyramid_rows(gy, K)
    last = {(k, R): min(2 ** k * (R + 1), gy) - 1 for k, R in order}
    encoded, groups = [], []

    def encode(run):
        assert 1 <= len(run) <= batch and run.shape[1:] == (ps, ps, 3)
        encoded.append(len(run))
        return torch.zeros((len(run), 2, 5), dtype=torch.int32)

    w = _Recorder((Y, X, 3), ps, K, batch, 'cpu', lambda k, idx: (k,) + idx, encode,
                  lambda sym, paths: groups.append((tuple(sym.shape), list(paths))), (2, 5))
    tiles = torch.zeros((batch, ps, ps, 3), dtype=torch.uint8)
    ij = np.array([(i, j) for i in range(gy) for j in range(gx)])
    for k0 in range(0, len(ij), batch):                         # batches span chunk rows
        w.add(tiles, ij[k0:k0 + batch])
    w.finish()
    assert w.flushed == order
    # a row is reduced after every level row it does not feed was flushed, before any it feeds
    assert sum(n for _, _, n in w.launches) == gy * gx
    for i, flushed, _ in w.launches:
        assert flushed == [o for o in order if last[o] < i], i
    # the groups: the default schedule over every level chunk, in pyramid_rows order
    want_paths = [(k, R, col, 0) for k, R in order for col in range(-(-gx // 2 ** k))]
    assert [p for _, ps_ in groups for p in ps_] == want_paths == w.paths
    sizes = _slide.group_sizes(len(want_paths), _slide.default_schedule(len(want_paths), batch),
                               batch)
    assert [len(p) for _, p in groups] == sizes
    assert [s[0] for s, _ in groups] == sizes and all(s[1:] == (2, 5) for s, _ in groups)
    assert sum(encoded) == len(want_paths)
    # whole batches, except at the end of a group
    ends = set(np.cumsum(sizes).tolist())
    assert all(n == batch or int(np.sum(encoded[:e + 1])) in ends for e, n in enumerate(encoded))
