"""Layer-by-layer tests of the convolution kernels (cae_conv_igemm, cae_conv_head,
cae_conv_direct and the layout kernels) against a float64 reference built on the oracle's own
layer op, across the schedules, shapes and epilogues the kernels implement.

The reference is fed exactly the operands a kernel sees (fp16 activations, fp16 weights with
the BatchNorm scale folded in fp32 first) and emulates the epilogue at the kernel's rounding
points, so the tolerance is derived, not tuned:

  per element   |got - ref| <= ulp16(|ref|) + 2^-15 * S      (fp16 outputs)
                |got - ref| <= 2^-15 * S                      (fp32 latents)
  whole tensor  ||got - ref|| / ||ref|| <= 2^-11              (fp16 outputs)

with S = conv(|x|, |w|) + |b| (+ |skip|): one flip of the final fp16 rounding, plus fp32
against fp64 accumulation.  Every output buffer is filled with a sentinel before the call, so
stores outside the logical tensor (halo ring, COL_PAD units, padded channels, past the end)
are caught; every call is repeated with NaN in the input's COL_PAD units, which no output may
depend on.

The unmarked tests at the top check the layout helpers and the epilogue emulation on the CPU.
Set CAE_CONV_LAYERS_LOG to a file path to get the largest err / allowance ratio per group.
"""
import ctypes
import json
import math
import os
import subprocess
import sys
from collections import namedtuple
from dataclasses import dataclass, replace

import pytest
import torch
import torch.nn.functional as F

from cnn_autoencoder_b200 import _cabi as C
from cnn_autoencoder_b200 import _ops
from oracle import cae_oracle as O

PLANAR, SPLIT, F32, U8 = C.FMT_F16_PLANAR, C.FMT_F16_SPLIT, C.FMT_F32_NCHW, C.FMT_U8_HWC
KEEP, REFLECT = C.HALO_KEEP, C.HALO_REFLECT
NONE, LEAKY, RELU = C.ACT_NONE, C.ACT_LEAKY_RELU, C.ACT_RELU
S1, S2, T1, T2 = C.CONV_S1, C.CONV_S2, C.CONVT_S1, C.CONVT_S2
COL_PAD = _ops.COL_PAD
SLOPE = {NONE: 1.0, LEAKY: 0.01, RELU: 0.0}

ACC = 2.0 ** -15         # fp32 against fp64 accumulation, relative to S (tensor-core paths)
ACC_F32 = 2.0 ** -20     # the same for the CUDA-core fp32 paths (direct kernel)
REL_L2 = 2.0 ** -11

SENT16 = 0x7E5A          # a NaN payload no kernel computes
SENT32 = 0x7FA5A5A5
SENT8 = 0xA5
GUARD = 64               # guard elements before and after every fp32 / uint8 / fp16 output

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


# ------------------------------------------------------------------ layout helpers
def _planes(t, fmt):
    return t.shape[-4]


def pack_layout(x, fmt, halo, planes=None, col_fill=0.0):
    """(n, c, h, w) float -> fp16 tensor in the PLANAR ([N][C/8][H+2][W+8][8]) or SPLIT
    ([N][4][C/8][(H+2)/2][(W+8)/2][8]) layout of include/cae_b200.h.  Padded pixel (Y, X) sits at
    row Y, column X + CAE_COL_PAD; in SPLIT it lives in parity plane (Y&1)*2 + ((X+3)&1) at
    (Y>>1, (X+3)>>1).  halo KEEP: zero ring; REFLECT: mirrored interior.  Padded channels are 0,
    the COL_PAD units hold ``col_fill``."""
    n, c, h, w = x.shape
    p = planes or _ops.planes_for(c)
    padded = torch.zeros((n, p * 8, h + 2, w + 2), dtype=torch.float32)
    xf = x.float().cpu()
    if halo == REFLECT:
        padded[:, :c] = F.pad(xf, (1, 1, 1, 1), mode='reflect')
    else:
        padded[:, :c, 1:h + 1, 1:w + 1] = xf
    phys = torch.full((n, p * 8, h + 2, w + 2 + 2 * COL_PAD), col_fill, dtype=torch.float32)
    phys[..., COL_PAD:COL_PAD + w + 2] = padded
    phys = phys.half()
    hp, wp = h + 2, w + 2 + 2 * COL_PAD
    t = phys.reshape(n, p, 8, hp, wp)
    if fmt == PLANAR:
        return t.permute(0, 1, 3, 4, 2).contiguous()
    assert fmt == SPLIT and h % 2 == 0 and w % 2 == 0
    t = t.reshape(n, p, 8, hp // 2, 2, wp // 2, 2)          # Y = 2 Yh + py, Xc = 2 Xh + px
    return t.permute(0, 4, 6, 1, 3, 5, 2).reshape(n, 4, p, hp // 2, wp // 2, 8).contiguous()


Unpacked = namedtuple('Unpacked', 'interior padded halo col_pad chan_pad')


def halo_mask(h, w):
    m = torch.ones((h + 2, w + 2), dtype=torch.bool)
    m[1:h + 1, 1:w + 1] = False
    return m


def unpack_layout(t, fmt, n, c, h, w):
    """Inverse of pack_layout on any element type (an int16 view gives bit patterns):
    interior (n, c, h, w), the padded tensor with its halo (n, planes*8, h+2, w+2), the halo ring
    (n, planes*8, ring), the COL_PAD units (n, planes*8, h+2, 6) and the padded channels of the
    interior (n, planes*8 - c, h, w)."""
    t = t.cpu()
    p = _planes(t, fmt)
    hp, wp = h + 2, w + 2 + 2 * COL_PAD
    if fmt == PLANAR:
        phys = t.reshape(n, p, hp, wp, 8).permute(0, 1, 4, 2, 3).reshape(n, p * 8, hp, wp)
    else:
        phys = t.reshape(n, 2, 2, p, hp // 2, wp // 2, 8).permute(0, 3, 6, 4, 1, 5, 2)
        phys = phys.reshape(n, p * 8, hp, wp)
    padded = phys[..., COL_PAD:COL_PAD + w + 2]
    col_pad = torch.cat([phys[..., :COL_PAD], phys[..., COL_PAD + w + 2:]], dim=-1)
    return Unpacked(padded[:, :c, 1:h + 1, 1:w + 1], padded, padded[..., halo_mask(h, w)],
                    col_pad, padded[:, c:, 1:h + 1, 1:w + 1])


# ------------------------------------------------------------------ reference
def _stride(kind):
    return 2 if kind in (S2, T2) else 1


def _transposed(kind):
    return kind in (T1, T2)


def _conv64(kind, x, w, b, pad_mode, groups):
    """One layer through the oracle's op ('conv' reflect-padded, 'convT' with output_padding =
    stride - 1); only the zero-padded Conv2d of the head / direct kernels is spelled out."""
    tr = _transposed(kind)
    cin = x.shape[1]
    cout = (w.shape[1] * (cin if groups else 1)) if tr else w.shape[0]
    if not tr and pad_mode == C.PAD_ZERO:
        return F.conv2d(x, w, b, stride=_stride(kind), padding=1, groups=cin if groups else 1)
    sd = {'l.weight': w}
    if b is not None:
        sd['l.bias'] = b
    op = ('convT' if tr else 'conv', 'l', cin, cout, _stride(kind))
    return O._apply_op(x, op, sd, groups, 'analysis')


def kernel_weights(kind, w, scale=None, f16=True):
    """The weights a kernel multiplies with: w * scale per output channel in fp32
    (pack_weights_kernel), then rounded to fp16 (__float2half_rn) on the tensor-core paths."""
    w = w.float()
    if scale is not None:
        s = scale.float()
        w = w * (s.reshape(1, -1, 1, 1) if _transposed(kind) else s.reshape(-1, 1, 1, 1))
    return w.half().double() if f16 else w.double()


def ref_conv(kind, x, w, b=None, scale=None, pre=NONE, post=NONE, skip=None,
             pad_mode=C.PAD_REFLECT, groups=False, path='fast'):
    """float64 reference of one kernel call: returns (out, S, z).  x / skip are the values the
    kernel reads (already fp16 where it reads fp16), w the fp32 torch-layout weights; the
    tensor-core paths see w * scale rounded to fp16.  z = conv + bias, out = the epilogue
    emulated on ``path``; S = conv(|x|, |w|) + |b| (+ |skip|)."""
    f16 = path != 'exact'
    w64 = kernel_weights(kind, w, scale, f16)
    x64 = x.double()
    b64 = b.double() if b is not None else None
    z = _conv64(kind, x64, w64, b64, pad_mode, groups)
    S = _conv64(kind, x64.abs(), w64.abs(), b64.abs() if b is not None else None, pad_mode, groups)
    sk = skip.double() if skip is not None else None
    if sk is not None:
        S = S + sk.abs()
    return emulate_epilogue(z, pre, post, sk, path), S, z


def _act64(v, act):
    return torch.maximum(v, v * SLOPE[act])


def _act16(v, act):
    s16 = float(torch.tensor(SLOPE[act]).half())
    return torch.maximum(v, (v.double() * s16).half())


def emulate_epilogue(z, pre, post, skip=None, path='fast'):
    """igemm_conv.cu's epilogue at its rounding points.
    fast (planar / split, no skip): bias in fp32, round to fp16, each activation in fp16 as
        max(v, v * slope) (__hmax2 / __hmul2);
    residual (planar / split with skip): bias, pre-activation and skip add in fp32, round to
        fp16, post-activation in fp16;
    latent / image / exact: all fp32 (image: the caller truncates to uint8) -- 'exact' is the
        oracle's op sequence with every rounding point switched off."""
    if path == 'fast' and skip is None:
        return _act16(_act16(z.half(), pre), post).double()
    if path in ('fast', 'residual'):
        v = _act64(z, pre) + (skip if skip is not None else 0.0)
        return _act16(v.half(), post).double()
    v = _act64(z, pre)
    if skip is not None:
        v = v + skip
    return _act64(v, post)


def ulp16(a):
    """Spacing of fp16 numbers at |a| (2^-24 in the subnormal range)."""
    a = a.double().abs().clamp_min(2.0 ** -14)
    return torch.exp2(torch.floor(torch.log2(a)) - 10)


def scaled_flip(z, pre, post, skip=None, path='fast'):
    """An fp16 rounding flip at a point that an activation later scales: on the fast path
    fp16(z) and fp16(v * slope_pre) precede the fp16 activations, on the residual path fp16(v)
    precedes the post-activation.  A flip of one ulp there reaches the output multiplied by the
    slopes applied after it (LeakyReLU on a negative value); a flip that no activation scales is
    the final rounding, which ulp16(|ref|) already covers."""
    zero = torch.zeros_like(z)
    if path == 'fast' and skip is None:
        v0 = z.half().double()
        g_pre = torch.where(v0 < 0, SLOPE[pre], 1.0) if pre != NONE else torch.ones_like(z)
        v1 = _act16(z.half(), pre).double()
        g_post = torch.where(v1 < 0, SLOPE[post], 1.0) if post != NONE else torch.ones_like(z)
        g0 = g_pre * g_post
        t = torch.where(g0 != 1.0, ulp16(v0) * g0, zero)
        if pre != NONE:
            t = t + torch.where((g_pre != 1.0) & (g_post != 1.0), ulp16(v1) * g_post, zero)
        return t
    if path in ('fast', 'residual') and post != NONE:
        v = (_act64(z, pre) + (skip if skip is not None else 0.0)).half().double()
        g = torch.where(v < 0, SLOPE[post], 1.0)
        return torch.where(g != 1.0, ulp16(v) * g, zero)
    return zero


# ------------------------------------------------------------------ result bookkeeping
RATIOS = {}


def _note(group, ratio):
    RATIOS[group] = max(RATIOS.get(group, 0.0), float(ratio))


@pytest.fixture(scope='module', autouse=True)
def _ratio_log():
    yield
    path = os.environ.get('CAE_CONV_LAYERS_LOG')
    if path and RATIOS:
        with open(path, 'a') as f:
            f.write(json.dumps({k: round(v, 4) for k, v in sorted(RATIOS.items())}) + '\n')


def check_close(group, what, got, ref, allow, rel_l2=None):
    got, ref, allow = got.double(), ref.double(), allow.double()
    err = (got - ref).abs()
    r = err / allow
    worst = r.max().item() if r.numel() else 0.0
    _note(group, worst)
    if not worst <= 1.0:
        i = int(torch.nan_to_num(r, nan=float('inf')).flatten().argmax())
        idx = tuple(int(v) for v in torch.unravel_index(torch.tensor(i), r.shape))
        raise AssertionError(f'{what}: worst err/allowance {worst:.3g} at {idx}: got '
                             f'{got.flatten()[i].item():.6g} ref {ref.flatten()[i].item():.6g} '
                             f'allowance {allow.flatten()[i].item():.3g}; '
                             f'{int((r > 1).sum())} of {r.numel()} elements over')
    if rel_l2 is not None and ref.norm() > 0:
        rel = ((got - ref).norm() / ref.norm()).item()
        assert rel <= rel_l2, f'{what}: relative L2 error {rel:.3g} > {rel_l2:.3g}'


def u8_report(u8, ref, bound):
    """Like test_gpu_parity._symbol_report for the image cast: (agreeing fraction, number of
    differing values, largest distance of a differing ref * 255 from an integer boundary in
    units of the allowance).  A correct kernel differs by at most 1 and only where ref * 255 lies
    within 255 * bound of an integer."""
    want = (ref * 255).clamp(0, 255).floor()
    d = (u8.double() - want)
    diff = d != 0
    s = (ref * 255).clamp(0, 255)
    dist = (s - torch.round(s)).abs() / (255 * bound)
    worst = dist[diff].max().item() if diff.any() else 0.0
    return 1 - diff.double().mean().item(), int(diff.sum()), worst, d.abs().max().item()


def check_u8(group, what, u8, ref, bound):
    agree, nflip, worst, dmax = u8_report(u8, ref, bound)
    _note(group + '/u8_boundary', worst)
    assert dmax <= 1 and worst <= 1.0, (what, agree, nflip, worst, dmax)


# ------------------------------------------------------------------ device buffers
def _bits_dtype(dtype):
    return {torch.float16: torch.int16, torch.float32: torch.int32, torch.uint8: torch.uint8,
            torch.int32: torch.int32, torch.float64: torch.int64}[dtype]


def _sentinel(dtype):
    return {torch.float16: SENT16, torch.float32: SENT32, torch.uint8: SENT8}[dtype]


def guarded(shape, dtype):
    """A sentinel-filled device buffer with GUARD elements before and after ``shape``."""
    numel = math.prod(shape)
    buf = torch.empty(numel + 2 * GUARD, dtype=dtype, device='cuda')
    buf.view(_bits_dtype(dtype)).fill_(_sentinel(dtype))
    return buf, buf[GUARD:GUARD + numel].view(shape)


def guards_intact(buf):
    b = buf.view(_bits_dtype(buf.dtype)).cpu()
    s = _sentinel(buf.dtype)
    return bool((b[:GUARD] == s).all()) and bool((b[-GUARD:] == s).all())


def out_act(fmt, n, c, h, w, halo=KEEP, planes=None):
    """Sentinel-filled output Act (planar / split / fp32 NCHW / uint8 HWC) inside guard bands."""
    shape = tuple(_ops.alloc_act(fmt, 1, c, h, w, device='meta', planes=planes).t.shape[1:])
    dtype = {PLANAR: torch.float16, SPLIT: torch.float16, F32: torch.float32, U8: torch.uint8}[fmt]
    buf, t = guarded((n,) + shape, dtype)
    return buf, _ops.Act(t, fmt, n, c, h, w, halo)


def in_act(x, fmt, halo=KEEP, col_fill=0.0, planes=None):
    n, c, h, w = x.shape
    if fmt in (PLANAR, SPLIT):
        t = pack_layout(x, fmt, halo, planes=planes, col_fill=col_fill).cuda()
    elif fmt == F32:
        t = x.float().contiguous().cuda()
    else:
        t = x.permute(0, 2, 3, 1).contiguous().cuda()
    return _ops.Act(t, fmt, n, c, h, w)


def check_act_output(group, what, buf, act, ref, allow, n, c, h, w, halo, rel=True,
                     padded_planes_written=True):
    """Interior against the reference; padded channels +0; halo ring mirrored (REFLECT) or
    untouched (KEEP); COL_PAD units and guard bands untouched."""
    bits = act.t.view(torch.int16)
    ub = unpack_layout(bits, act.fmt, n, c, h, w)
    got = ub.interior.view(torch.float16)
    check_close(group, what, got, ref, allow, REL_L2 if rel else None)
    p8 = act.planes * 8
    c_written = p8 if padded_planes_written else (c + 7) // 8 * 8
    assert (ub.chan_pad[:, :c_written - c] == 0).all(), f'{what}: padded channels are not +0'
    if c_written < p8:
        assert (ub.chan_pad[:, c_written - c:] == SENT16).all(), f'{what}: store into an unused plane'
    assert (ub.col_pad == SENT16).all(), f'{what}: store into the COL_PAD units'
    assert guards_intact(buf), f'{what}: store outside the buffer'
    ring = ub.padded[:, :c_written]
    if halo == REFLECT:
        inner = ring[:, :, 1:h + 1, 1:w + 1].float()
        want = F.pad(inner, (1, 1, 1, 1), mode='reflect').to(torch.int16)
        assert torch.equal(ring, want), f'{what}: reflect halo is not the mirrored interior'
    else:
        assert (ub.halo == SENT16).all(), f'{what}: store into the halo of a HALO_KEEP output'


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _randn(g, *shape, s=1.0):
    return torch.randn(*shape, generator=g) * s


def _weights(g, kind, c_in, c_out, groups=False, gain=1.0):
    per = c_in if groups else 1
    shape = (c_in, c_out // per, 3, 3) if _transposed(kind) else (c_out, c_in // per, 3, 3)
    return _randn(g, *shape, s=gain / math.sqrt(9 * (c_in // per)))


def _out_size(kind, h, w):
    return _ops.KIND_OUT[kind](h, w)


# ------------------------------------------------------------------ CPU tests of the helpers
@pytest.mark.parametrize('fmt', [PLANAR, SPLIT])
@pytest.mark.parametrize('h,w', [(2, 2), (4, 6), (3, 5), (10, 7), (1, 1)])
@pytest.mark.parametrize('halo', [KEEP, REFLECT])
def test_pack_unpack_round_trip_and_shapes(fmt, h, w, halo):
    if fmt == SPLIT and (h % 2 or w % 2):
        pytest.skip('split layout needs even sizes')
    if halo == REFLECT and min(h, w) < 2:
        pytest.skip('reflect padding needs size >= 2')
    g = _gen(h * 100 + w)
    for c in (1, 8, 20):
        x = _randn(g, 2, c, h, w).half().float()
        t = pack_layout(x, fmt, halo, col_fill=float('nan'))
        assert t.shape == _ops.alloc_act(fmt, 2, c, h, w, device='cpu').t.shape
        u = unpack_layout(t, fmt, 2, c, h, w)
        assert torch.equal(u.interior.float(), x)
        assert (u.chan_pad == 0).all() and torch.isnan(u.col_pad).all()
        want = F.pad(x, (1, 1, 1, 1), mode='reflect') if halo == REFLECT else F.pad(x, (1, 1, 1, 1))
        assert torch.equal(u.padded[:, :c].float(), want)
        assert u.halo.shape[-1] == 2 * (h + 2) + 2 * w


def test_pixel_origin_sits_at_column_four():
    x = torch.zeros(1, 8, 2, 2)
    x[0, 3, 0, 0] = 1.0
    t = pack_layout(x, PLANAR, KEEP)
    assert t[0, 0, 1, 4, 3] == 1 and t.float().sum() == 1        # row Y = 1, column X + 3 = 4
    s = pack_layout(x, SPLIT, KEEP)
    # padded (1, 1): parity (1 & 1) * 2 + ((1 + 3) & 1) = 2, at (0, 2)
    assert s[0, 2, 0, 0, 2, 3] == 1 and s.float().sum() == 1


def test_layout_helpers_match_the_documented_strides():
    """Unit offset of (n, plane, Y, X) as cae_common.cuh's act_unit_offset computes it."""
    n, c, h, w = 2, 24, 6, 4
    x = torch.arange(n * c * h * w, dtype=torch.float32).reshape(n, c, h, w) % 1000
    for fmt in (PLANAR, SPLIT):
        t = pack_layout(x, fmt, KEEP)
        flat = t.reshape(-1, 8)
        p = _ops.planes_for(c)
        rows = w + 2 + 2 * COL_PAD
        for (ni, ci, y, xx) in ((0, 0, 0, 0), (1, 17, 5, 3), (1, 9, 2, 1), (0, 23, 4, 0)):
            Y, X = y + 1, xx + 1
            if fmt == PLANAR:
                u = ((ni * p + ci // 8) * (h + 2) + Y) * rows + X + COL_PAD
            else:
                Xc = X + COL_PAD
                par = ((Y & 1) << 1) | (Xc & 1)
                u = (((ni * 4 + par) * p + ci // 8) * ((h + 2) // 2) + (Y >> 1)) * (rows // 2) + (Xc >> 1)
            assert flat[u, ci % 8].item() == x[ni, ci, y, xx].item()


@pytest.mark.parametrize('pre,post', [(NONE, NONE), (LEAKY, NONE), (NONE, RELU), (LEAKY, LEAKY),
                                      (RELU, LEAKY)])
def test_epilogue_emulation_without_rounding_is_the_oracle(pre, post):
    g = _gen(5)
    name = {NONE: None, LEAKY: 'LeakyReLU', RELU: 'ReLU'}
    x = _randn(g, 2, 5, 6, 7).double()
    w = _randn(g, 4, 5, 3, 3)
    b = _randn(g, 4)
    skip = _randn(g, 2, 4, 6, 7).double()
    for sk in (None, skip):
        out, S, z = ref_conv(S1, x, w, b, None, pre, post, sk, path='exact')
        want = O._apply_op(x, ('conv', 'l', 5, 4, 1), {'l.weight': w.double(), 'l.bias': b.double()},
                           False, 'analysis')
        want = O._apply_act(want, name[pre], {}, '', 'analysis')
        if sk is not None:
            want = want + sk
        want = O._apply_act(want, name[post], {}, '', 'analysis')
        assert torch.allclose(out, want, rtol=0, atol=1e-12)
    # with the rounding points on, the fast path is fp16(z) for identity activations
    out, _, z = ref_conv(S1, x, w, b, None, NONE, NONE, None, path='fast')
    assert torch.equal(out, z.half().double())


def test_reference_transposed_and_grouped_forms():
    """convT of the reference = the adjoint of conv; groups=True = per-channel convolutions."""
    g = _gen(9)
    x = _randn(g, 1, 3, 5, 4).double()
    w = _randn(g, 3, 6, 3, 3).double()
    for kind, size in ((T1, (5, 4)), (T2, (10, 8))):
        out, S, _ = ref_conv(kind, x, w.float(), path='exact')
        assert out.shape[-2:] == size
        assert (S + 1e-12 >= out.abs()).all()
    out, _, _ = ref_conv(S1, x, _randn(g, 3, 1, 3, 3), groups=True, path='exact')
    assert out.shape == (1, 3, 5, 4)


def test_ulp16_and_scaled_flip():
    assert ulp16(torch.tensor([1.0, 1.5, 2.0, 0.0, 2.0 ** -20])).tolist() == \
        [2.0 ** -10, 2.0 ** -10, 2.0 ** -9, 2.0 ** -24, 2.0 ** -24]
    z = torch.tensor([-4.0, 4.0], dtype=torch.float64)
    t = scaled_flip(z, LEAKY, NONE)
    assert t[1] == 0 and abs(t[0].item() - 0.01 * 2.0 ** -8) < 1e-12
    assert (scaled_flip(z, RELU, NONE) == 0).all()


# ================================================================== cae_conv_igemm
@dataclass
class IgCase:
    kind: int
    c_in: int
    c_out: int
    n: int
    h: int
    w: int
    out: str = 'planar'        # planar | split | f32 | u8 | u8+aux | aux
    halo: int = KEEP
    ck: int = 0
    mt: int = 0
    grid: int = 0
    bias: bool = True
    pre: int = NONE
    post: int = NONE
    skip: int = 0              # 0, PLANAR or SPLIT
    scale: bool = False
    refused: bool = False      # a legal ck whose stages do not fit shared memory: CAE_CHECK
    seed: int = 0

    @property
    def id(self):
        k = {S1: 's1', S2: 's2', T1: 't1', T2: 't2'}[self.kind]
        s = f'{k}_{self.c_in}-{self.c_out}_n{self.n}_{self.h}x{self.w}_{self.out}'
        s += {KEEP: '', REFLECT: '_refl'}[self.halo]
        for name, v in (('ck', self.ck), ('mt', self.mt), ('grid', self.grid)):
            if v:
                s += f'_{name}{v}'
        if self.pre or self.post:
            s += f'_a{self.pre}{self.post}'
        if self.skip:
            s += '_skip' + ('P' if self.skip == PLANAR else 'S')
        if self.scale:
            s += '_bn'
        if not self.bias:
            s += '_nobias'
        return s + ('_refused' if self.refused else '')


def _legal_cks(c_in):
    cp = (c_in + 15) // 16 * 16
    return [ck for ck in (16, 32, 48, 64, 128) if cp % ck == 0]


# (kind, c_in, ck) that pack but whose activation stage next to two weight stages exceeds the
# shared memory of an SM: the launcher refuses them before anything is launched
REFUSED_CK = {(S1, 128, 128), (S1, 256, 128), (S2, 128, 64), (S2, 128, 128)}


def _ig_cases():
    c = [
        # CONV_S1: every auto_ck branch (16, 32, 48, 64) and N = 16 .. 256
        IgCase(S1, 8, 16, 1, 2, 2, pre=LEAKY),
        IgCase(S1, 24, 40, 2, 18, 10, out='split', halo=REFLECT, mt=1, bias=False, post=RELU, scale=True),
        IgCase(S1, 48, 48, 3, 34, 70, halo=REFLECT, skip=PLANAR, pre=LEAKY, post=LEAKY),
        IgCase(S1, 48, 48, 1, 34, 70, out='split', skip=SPLIT, grid=3, post=LEAKY),
        IgCase(S1, 64, 128, 1, 64, 96, grid=1, mt=2, post=LEAKY),          # 24 tiles on one CTA
        IgCase(S1, 64, 128, 2, 17, 9, out='f32', mt=1, pre=RELU),
        IgCase(S1, 128, 192, 1, 20, 24, halo=REFLECT, scale=True, pre=LEAKY),
        IgCase(S1, 128, 192, 1, 8, 8, out='f32', post=LEAKY),              # dom_w <= 8
        IgCase(S1, 256, 256, 1, 18, 10, halo=REFLECT, skip=PLANAR, post=LEAKY),
        IgCase(S1, 256, 256, 2, 6, 5, out='f32', grid=1, scale=True),
        # CONV_S2 (split input)
        IgCase(S2, 16, 32, 1, 2, 2),                                        # smallest: 1 x 1 out
        IgCase(S2, 40, 24, 2, 36, 20, out='split', halo=REFLECT, pre=RELU),
        IgCase(S2, 48, 128, 3, 68, 140, grid=3, mt=1, post=LEAKY, scale=True),
        IgCase(S2, 48, 128, 1, 68, 140, halo=REFLECT, mt=2, skip=SPLIT, pre=LEAKY, post=RELU),
        IgCase(S2, 128, 48, 2, 36, 20, out='f32', post=LEAKY),             # the latent layer
        IgCase(S2, 128, 48, 1, 4, 2, out='f32', bias=False),
        IgCase(S2, 128, 192, 1, 16, 16, halo=REFLECT, skip=PLANAR, post=LEAKY),
        IgCase(S2, 128, 192, 2, 40, 68, grid=1, pre=LEAKY),
        # CONVT_S1 (zero halo input)
        IgCase(T1, 48, 48, 2, 18, 10, halo=REFLECT, skip=PLANAR, pre=LEAKY, post=RELU),
        IgCase(T1, 192, 128, 1, 34, 70, out='split', post=LEAKY, scale=True),
        IgCase(T1, 192, 128, 3, 7, 5, grid=1, bias=False),
        # CONVT_S2: one pass (4 N <= 256) and two passes
        IgCase(T2, 16, 16, 1, 1, 1),
        IgCase(T2, 16, 16, 2, 9, 17, halo=REFLECT, pre=LEAKY, grid=3),
        IgCase(T2, 32, 64, 2, 9, 5, halo=REFLECT, skip=PLANAR, post=LEAKY),
        IgCase(T2, 32, 64, 1, 16, 24, out='split', grid=1),
        IgCase(T2, 48, 128, 1, 17, 35, post=LEAKY, scale=True),
        IgCase(T2, 48, 128, 2, 8, 12, out='split', halo=REFLECT, mt=1, pre=RELU),
        IgCase(T2, 128, 128, 1, 16, 32, out='split', halo=REFLECT, grid=1, post=LEAKY),
        IgCase(T2, 128, 128, 2, 5, 9, skip=SPLIT, pre=LEAKY, post=LEAKY),
        IgCase(T2, 256, 256, 1, 5, 9, halo=REFLECT, skip=PLANAR, post=LEAKY),
        IgCase(T2, 256, 256, 1, 3, 2, out='split', bias=False),
        # the merged image layer (c_out <= 4)
        IgCase(T2, 128, 1, 2, 9, 17, out='u8+aux'),
        IgCase(T2, 128, 2, 1, 8, 8, out='u8', post=RELU, grid=1),
        IgCase(T2, 128, 3, 2, 17, 33, out='u8+aux', pre=LEAKY, scale=True),
        IgCase(T2, 128, 3, 1, 1, 1, out='aux'),
        IgCase(T2, 128, 4, 2, 9, 5, out='u8+aux', post=LEAKY),
        IgCase(T2, 64, 2, 1, 12, 20, out='u8+aux', mt=1),
    ]
    # every legal forced ck on one layer of each kind (pack and launch with the same ck)
    for base in (IgCase(S1, 64, 128, 1, 34, 70, halo=REFLECT, post=LEAKY),
                 IgCase(S1, 128, 192, 1, 18, 10, post=LEAKY),
                 IgCase(S1, 256, 256, 1, 9, 17, grid=3),
                 IgCase(S2, 40, 24, 1, 20, 36),
                 IgCase(S2, 128, 48, 1, 20, 36, out='f32'),
                 IgCase(T1, 192, 128, 1, 18, 10, skip=PLANAR),
                 IgCase(T2, 128, 128, 1, 9, 17, post=LEAKY),
                 IgCase(T2, 128, 3, 1, 9, 17, out='u8+aux')):
        for ck in _legal_cks(base.c_in):
            c.append(replace(base, ck=ck, refused=(base.kind, base.c_in, ck) in REFUSED_CK))
    for i, case in enumerate(c):
        case.seed = 1000 + i
    return c


IG_CASES = _ig_cases()


def _group(case):
    if case.out in ('f32',):
        return 'igemm/latent'
    if case.out in ('u8', 'u8+aux', 'aux'):
        return 'igemm/image'
    return 'igemm/residual' if case.skip else 'igemm/fast'


def _ig_operands(case):
    g = _gen(case.seed)
    image = case.out in ('u8', 'u8+aux', 'aux')
    x = _randn(g, case.n, case.c_in, case.h, case.w).half().float()
    w = _weights(g, case.kind, case.c_in, case.c_out, gain=0.3 if image else 1.0)
    b = (_randn(g, case.c_out, s=0.2) + (0.5 if image else 0.0)) if case.bias else None
    scale = None
    if case.scale:
        scale = (torch.rand(case.c_out, generator=g) * 1.5 + 0.25) * \
            torch.where(torch.rand(case.c_out, generator=g) < 0.3, -1.0, 1.0)
    oh, ow = _out_size(case.kind, case.h, case.w)
    skip = _randn(g, case.n, case.c_out, oh, ow, s=0.5).half().float() if case.skip else None
    return x, w, b, scale, skip


def run_igemm(case, col_fill, x, packed, b, skip):
    """One cae_conv_igemm call on freshly sentinel-filled outputs; returns the buffers."""
    oh, ow = _out_size(case.kind, case.h, case.w)
    in_fmt = SPLIT if case.kind == S2 else PLANAR
    in_halo = REFLECT if case.kind in (S1, S2) else KEEP
    xa = in_act(x, in_fmt, in_halo, col_fill=col_fill)
    sk = in_act(skip, case.skip, KEEP) if case.skip else None
    bufs = {}
    out = aux = None
    if case.out in ('planar', 'split'):
        buf, out = out_act(PLANAR if case.out == 'planar' else SPLIT, case.n, case.c_out, oh, ow, case.halo)
        bufs['out'] = (buf, out)
    elif case.out == 'f32':
        buf, out = out_act(F32, case.n, case.c_out, oh, ow)
        bufs['out'] = (buf, out)
    else:
        if 'u8' in case.out:
            buf, out = out_act(U8, case.n, case.c_out, oh, ow)
            bufs['out'] = (buf, out)
        if 'aux' in case.out:
            abuf, aux = guarded((case.n, case.c_out, oh, ow), torch.float32)
            bufs['aux'] = (abuf, aux)
    _ops.conv(case.kind, xa, packed, case.c_out, out, igemm=True,
              bias=b.cuda() if b is not None else None, skip=sk, pre_act=case.pre,
              post_act=case.post, aux=aux, ck=case.ck, mt=case.mt, grid=case.grid)
    torch.cuda.synchronize()
    return bufs


def _bits(buf):
    return buf.view(_bits_dtype(buf.dtype)).cpu()


def check_igemm_case(case):
    group = _group(case)
    x, w, b, scale, skip = _ig_operands(case)
    oh, ow = _out_size(case.kind, case.h, case.w)
    packed = _ops.pack_weights(case.kind, w.cuda(), scale.cuda() if scale is not None else None,
                               ck=case.ck)
    if case.refused:
        with pytest.raises(C.CaeError, match='does not fit shared memory'):
            run_igemm(case, 0.0, x, packed, b, skip)
        return
    first = run_igemm(case, 0.0, x, packed, b, skip)
    second = run_igemm(case, float('nan'), x, packed, b, skip)
    for k in first:
        assert torch.equal(_bits(first[k][0]), _bits(second[k][0])), \
            f'{case.id}: output {k} depends on the input COL_PAD units'
    path = {'igemm/latent': 'latent', 'igemm/image': 'image', 'igemm/fast': 'fast',
            'igemm/residual': 'residual'}[group]
    ref, S, z = ref_conv(case.kind, x, w, b, scale, case.pre, case.post, skip, path=path)
    if path in ('fast', 'residual'):
        buf, act = first['out']
        got = unpack_layout(act.t.view(torch.int16), act.fmt, case.n, case.c_out, oh, ow).interior
        sk = skip.double() if skip is not None else None
        allow = (ACC * S + torch.maximum(ulp16(ref), ulp16(got.view(torch.float16))) +
                 scaled_flip(z, case.pre, case.post, sk, path))
        check_act_output(group, case.id, buf, act, ref, allow, case.n, case.c_out, oh, ow, case.halo)
        return
    if path == 'latent':
        buf, act = first['out']
        check_close(group, case.id, act.t.cpu(), ref, ACC * S)
        assert guards_intact(buf), f'{case.id}: store outside the fp32 output'
        return
    # image layer: fp32 epilogue, truncating cast
    if 'aux' in first:
        abuf, aux = first['aux']
        check_close(group, case.id + ' aux', aux.cpu(), ref, ACC * S)
        assert guards_intact(abuf), f'{case.id}: store outside aux'
    if 'out' in first:
        buf, act = first['out']
        u8 = act.t.cpu().permute(0, 3, 1, 2)
        assert guards_intact(buf), f'{case.id}: store outside the uint8 image'
        if 'aux' in first:
            a = first['aux'][1].cpu()
            assert torch.equal(u8, (a * 255.0).clamp(0, 255).to(torch.uint8)), \
                f'{case.id}: uint8 output is not trunc(clip(aux * 255))'
        check_u8(group, case.id, u8, ref, ACC * S)


@pytest.mark.gpu
@pytest.mark.parametrize('case', IG_CASES, ids=[c.id for c in IG_CASES])
def test_igemm_layer_against_float64_reference(case):
    check_igemm_case(case)


# ------------------------------------------------------------------ fused quantizer
def _tables(c, g, lut_min=-150, lut_len=301):
    med = torch.rand(c, generator=g) * 4 - 2
    lut = torch.rand(c, lut_len, generator=g) * 0.5 + 1e-6
    return dict(medians=med.cuda(), lut=lut.cuda(), lut_min=lut_min, lut_len=lut_len)


def _abi_tables(tb):
    t = C.EbTables()
    t.medians = tb['medians'].data_ptr()
    t.lut = tb['lut'].data_ptr()
    t.lut_min, t.lut_len = tb['lut_min'], tb['lut_len']
    t.hist_min, t.hist_bins = tb['lut_min'], tb['lut_len']
    t.tail_lik = 1e-9          # the table ends where the likelihood bound begins
    t.lik_bound = 1e-9
    return t


def run_quant_layer(c_in, c_out, n, h, w, seed, col_fill):
    g = _gen(seed)
    x = _randn(g, n, c_in, h, w).half().float()
    wt = _weights(g, S2, c_in, c_out, gain=3.0)
    b = _randn(g, c_out, s=0.5)
    # channels whose symbols leave the shared-memory core window of the launcher (core symbols
    # around the median, as many as fit 40 KB) and channels whose symbols leave the likelihood
    # table (|sym| ~ 200 > 150)
    core = (40 * 1024 // (4 * c_out) - 1) // 2
    b[0:4] += core // 2 + 20
    b[4:8] -= core // 2 + 20
    b[8:10] += 200
    b[10:12] -= 200
    tb = _tables(c_out, g)
    packed = _ops.pack_weights(S2, wt.cuda())
    xa = in_act(x, SPLIT, REFLECT, col_fill=col_fill)
    oh, ow = h // 2, w // 2
    _, y = out_act(F32, n, c_out, oh, ow)
    q = C.QuantFuse()
    q.tables = _abi_tables(tb)
    res = dict(y=y.t,
               y_q=torch.empty((n, c_out, oh, ow), dtype=torch.float32, device='cuda'),
               sym=torch.empty((n, c_out, oh, ow), dtype=torch.int32, device='cuda'),
               planar=_ops.alloc_act(PLANAR, n, c_out, oh, ow),
               hist=torch.zeros((c_out, tb['lut_len']), dtype=torch.int32, device='cuda'),
               rate=torch.zeros(1, dtype=torch.float64, device='cuda'),
               status=torch.zeros(1, dtype=torch.int32, device='cuda'))
    q.y_q, q.symbols = res['y_q'].data_ptr(), res['sym'].data_ptr()
    q.y_q_planar = res['planar'].desc()
    q.hist, q.rate_bits, q.status = res['hist'].data_ptr(), res['rate'].data_ptr(), res['status'].data_ptr()
    _ops.conv(S2, xa, packed, c_out, y, igemm=True, bias=b.cuda(), quant=q)
    torch.cuda.synchronize()
    res['planar'] = res['planar'].t
    return res, (x, wt, b, tb)


def eb_quantize(y, tb):
    n, c = y.shape[:2]
    hw = y[0, 0].numel()
    t = _abi_tables(tb)
    out = dict(y_q=torch.empty_like(y), sym=torch.empty(y.shape, dtype=torch.int32, device='cuda'),
               hist=torch.zeros((c, tb['lut_len']), dtype=torch.int32, device='cuda'),
               rate=torch.zeros(1, dtype=torch.float64, device='cuda'),
               status=torch.zeros(1, dtype=torch.int32, device='cuda'))
    C.check(C.lib().cae_eb_quantize(y.data_ptr(), n, c, hw, ctypes.byref(t), out['y_q'].data_ptr(),
                                    None, out['sym'].data_ptr(), out['hist'].data_ptr(),
                                    out['rate'].data_ptr(), out['status'].data_ptr(),
                                    _ops._stream_ptr(y)))
    torch.cuda.synchronize()
    return out


def check_quant_layer(c_in=128, c_out=48, n=2, h=36, w=44, seed=7):
    a, (x, wt, b, tb) = run_quant_layer(c_in, c_out, n, h, w, seed, 0.0)
    bnan, _ = run_quant_layer(c_in, c_out, n, h, w, seed, float('nan'))
    for k in a:
        assert torch.equal(_bits(a[k]), _bits(bnan[k])), f'quant: {k} depends on the input COL_PAD units'
    ref, S, _ = ref_conv(S2, x, wt, b, path='latent')
    check_close('igemm/quant', 'quant latent', a['y'].cpu(), ref, ACC * S)
    s = eb_quantize(a['y'], tb)
    sym = s['sym'].cpu()
    lut_min, lut_len = tb['lut_min'], tb['lut_len']
    core = (40 * 1024 // (4 * c_out) - 1) // 2
    assert ((sym.abs() > core // 2 + 2) & (sym >= lut_min) & (sym < lut_min + lut_len)).any(), \
        'no symbol outside the shared-memory core'
    assert ((sym < lut_min) | (sym >= lut_min + lut_len)).any(), 'no symbol outside the table'
    assert torch.equal(a['sym'], s['sym'])
    assert torch.equal(a['y_q'], s['y_q'])
    want_pl = pack_layout(s['y_q'].cpu(), PLANAR, KEEP)
    assert torch.equal(a['planar'].cpu().view(torch.int16), want_pl.view(torch.int16))
    assert torch.equal(a['hist'], s['hist'])
    assert int(a['hist'].sum()) == a['y'].numel()
    assert int(a['status'].item()) == 0 and int(s['status'].item()) == 0
    r, rs = a['rate'].item(), s['rate'].item()
    assert abs(r - rs) <= 1e-5 * abs(rs), (r, rs)


@pytest.mark.gpu
@pytest.mark.parametrize('c_out,hw', [(48, (36, 44)), (24, (18, 70))])
def test_fused_quantizer_matches_the_standalone_quantizer(c_out, hw):
    check_quant_layer(c_out=c_out, h=hw[0], w=hw[1])


# ------------------------------------------------------------------ opt-in forms (child processes)
PAIR_CASES = [
    IgCase(S1, 64, 128, 2, 34, 70, halo=REFLECT, post=LEAKY, seed=1),
    IgCase(S1, 64, 128, 1, 17, 9, ck=16, grid=3, pre=RELU, scale=True, seed=2),
    IgCase(S1, 128, 128, 1, 18, 10, skip=PLANAR, post=LEAKY, seed=3),
    IgCase(S2, 48, 128, 2, 68, 140, pre=LEAKY, seed=4),
    IgCase(S2, 128, 128, 1, 16, 16, out='split', halo=REFLECT, seed=5),
    IgCase(T1, 192, 128, 1, 34, 70, out='split', post=LEAKY, seed=6),
    IgCase(T2, 48, 128, 1, 17, 35, post=LEAKY, seed=7),
    IgCase(T2, 128, 128, 2, 5, 9, skip=SPLIT, pre=LEAKY, post=LEAKY, seed=8),
    IgCase(T2, 128, 128, 1, 16, 32, halo=REFLECT, ck=32, grid=3, seed=9),
]


def child_main(what):
    if what == 'pair':
        for case in PAIR_CASES:
            check_igemm_case(case)
    else:
        check_quant_layer()
        check_quant_layer(c_out=24, h=18, w=70)
    print(json.dumps(RATIOS))


@pytest.mark.gpu
@pytest.mark.parametrize('env,what', [
    ({'CAE_IGEMM_PAIR_MMA': '1'}, 'pair'),
    ({'CAE_IGEMM_PAIR_MMA': '1', 'CAE_IGEMM_NO_RESIDENT': '1'}, 'pair'),
    ({'CAE_QUANT_NO_SMEM': '1'}, 'quant'),
], ids=['pair', 'pair_no_resident', 'quant_no_smem'])
def test_opt_in_forms_in_a_child_process(env, what):
    """Knobs are read once per process and honoured only with CAE_DEBUG=1."""
    e = {k: v for k, v in os.environ.items() if not k.startswith('CAE_IGEMM') and k != 'CAE_QUANT_NO_SMEM'}
    e.update(env, CAE_DEBUG='1')
    script = ('import sys; sys.path[:0] = [%r, %r]; import test_gpu_conv_layers as T; T.child_main(%r)'
              % (ROOT, HERE, what))
    r = subprocess.run([sys.executable, '-c', script], env=e, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    for k, v in json.loads(r.stdout.strip().splitlines()[-1]).items():
        _note(f'{k}[{"+".join(sorted(env))}]', v)


# ================================================================== cae_conv_head
@dataclass
class HeadCase:
    c_in: int
    c_out: int
    in_fmt: int
    pad: int
    residual: bool
    act_stem: int
    act_down: int
    act_mid: int
    n: int
    h: int
    w: int
    halo: int = KEEP
    bias: bool = True
    seed: int = 0

    @property
    def id(self):
        return (f'{self.c_in}-{self.c_out}_{"u8" if self.in_fmt == U8 else "f32"}_'
                f'{"refl" if self.pad == C.PAD_REFLECT else "zero"}{"_res" if self.residual else ""}_'
                f'a{self.act_stem}{self.act_down}{self.act_mid}_n{self.n}_{self.h}x{self.w}'
                f'{"_outrefl" if self.halo == REFLECT else ""}{"" if self.bias else "_nobias"}')


Z, R = C.PAD_ZERO, C.PAD_REFLECT
HEAD_CASES = [
    HeadCase(3, 16, U8, R, False, LEAKY, LEAKY, NONE, 1, 2, 2),
    HeadCase(1, 24, F32, Z, False, RELU, NONE, NONE, 2, 17, 65, halo=REFLECT),
    HeadCase(2, 48, U8, Z, True, LEAKY, RELU, LEAKY, 1, 33, 70),
    HeadCase(4, 128, F32, R, True, NONE, LEAKY, RELU, 2, 18, 66, halo=REFLECT),
    HeadCase(3, 128, U8, R, False, LEAKY, NONE, NONE, 1, 40, 72, halo=REFLECT),
    HeadCase(1, 16, U8, R, True, RELU, LEAKY, NONE, 3, 5, 3, halo=REFLECT),
    HeadCase(2, 24, F32, R, False, NONE, RELU, NONE, 1, 9, 130),
    HeadCase(4, 48, U8, Z, False, LEAKY, LEAKY, NONE, 2, 3, 2),
    HeadCase(3, 48, F32, Z, True, LEAKY, LEAKY, LEAKY, 1, 35, 67, halo=REFLECT),
    HeadCase(1, 128, F32, R, False, NONE, NONE, NONE, 1, 64, 64, bias=False),
    HeadCase(4, 16, U8, R, False, RELU, LEAKY, NONE, 1, 16, 128, halo=REFLECT),
    HeadCase(2, 128, U8, R, True, LEAKY, NONE, LEAKY, 2, 2, 2),
    HeadCase(3, 24, U8, Z, True, NONE, NONE, NONE, 1, 31, 33, halo=REFLECT, bias=False),
    HeadCase(4, 24, F32, Z, False, RELU, RELU, NONE, 1, 2, 2),
]
for _i, _c in enumerate(HEAD_CASES):
    _c.seed = 2000 + _i


def _stem_conv(x, w, b, pad):
    return _conv64(S1, x, w.double(), b.double() if b is not None else None, pad, False)


def head_reference(case, x, ws, bs, wd, bd, ws2, bs2):
    """float64 head: the stem (fp32 in the kernel) rounded to fp16 where it enters the MMA,
    then the stride-2 convolution with fp16 weights and the fast epilogue (fp16(z), act_down in
    fp16).  Returns (out, allowance)."""
    x = x.double()
    s = _act64(_stem_conv(x, ws, bs, case.pad), case.act_stem)
    if case.residual:
        s = _act64(_stem_conv(s, ws2, bs2, case.pad) + x, case.act_mid)
    stem16 = s.half().double()
    wd16 = wd.half().double()
    bd64 = bd.double() if bd is not None else None
    z = _conv64(S2, stem16, wd16, bd64, case.pad, False)
    S = _conv64(S2, stem16.abs(), wd16.abs(), bd64.abs() if bd64 is not None else None, case.pad, False)
    flip = _conv64(S2, ulp16(s), wd.double().abs(), None, case.pad, False)
    out = emulate_epilogue(z, NONE, case.act_down, None, 'fast')
    allow = ACC * S + flip + ulp16(out) + scaled_flip(z, NONE, case.act_down)
    return out, allow


@pytest.mark.gpu
@pytest.mark.parametrize('case', HEAD_CASES, ids=[c.id for c in HEAD_CASES])
def test_head_against_float64_reference(case):
    g = _gen(case.seed)
    ci, co = case.c_in, case.c_out
    u8 = torch.randint(0, 256, (case.n, ci, case.h, case.w), generator=g, dtype=torch.uint8)
    x = u8.float() / 255.0 if case.in_fmt == U8 else torch.rand(case.n, ci, case.h, case.w, generator=g)
    ws = _randn(g, ci, ci, 3, 3, s=0.5)
    bs = _randn(g, ci, s=0.1) if case.bias else None
    wd = _randn(g, co, ci, 3, 3, s=1.0 / math.sqrt(9 * ci))
    bd = _randn(g, co, s=0.1) if case.bias else None
    ws2 = _randn(g, ci, ci, 3, 3, s=0.5) if case.residual else None
    bs2 = _randn(g, ci, s=0.1) if (case.residual and case.bias) else None
    xa = in_act(u8 if case.in_fmt == U8 else x, case.in_fmt)
    oh, ow = (case.h + 1) // 2, (case.w + 1) // 2
    buf, out = out_act(PLANAR, case.n, co, oh, ow, case.halo)
    cu = lambda t: t.cuda() if t is not None else None
    _ops.conv_head(xa, cu(ws), cu(bs), cu(wd), cu(bd), co, out, act_stem=case.act_stem,
                   act_down=case.act_down, pad_mode=case.pad, w_stem2=cu(ws2), b_stem2=cu(bs2),
                   act_mid=case.act_mid)
    torch.cuda.synchronize()
    ref, allow = head_reference(case, x, ws, bs, wd, bd, ws2, bs2)
    check_act_output('head', case.id, buf, out, ref, allow, case.n, co, oh, ow, case.halo)


# ================================================================== cae_conv_direct
@dataclass
class DirectCase:
    kind: int
    c_in: int
    c_out: int
    groups: bool
    in_fmt: int
    out_fmt: int
    pad: int
    skip: int = 0            # 0, F32, PLANAR or U8
    aux: bool = False
    pre: int = NONE
    post: int = NONE
    n: int = 2
    h: int = 6
    w: int = 10
    seed: int = 0

    @property
    def id(self):
        f = {U8: 'u8', F32: 'f32', PLANAR: 'pl', SPLIT: 'sp', 0: ''}
        k = {S1: 's1', S2: 's2', T1: 't1', T2: 't2'}[self.kind]
        return (f'{k}_{self.c_in}-{self.c_out}{"_g" if self.groups else ""}_{f[self.in_fmt]}-'
                f'{f[self.out_fmt]}_{"refl" if self.pad == R else "zero"}'
                f'{"_skip" + f[self.skip] if self.skip else ""}{"_aux" if self.aux else ""}'
                f'_a{self.pre}{self.post}_{self.h}x{self.w}')


def _direct_cases():
    fmts = [U8, F32, PLANAR, SPLIT]
    kinds = [S1, S2, T1, T2]
    chans = [(1, 1), (3, 3), (4, 8), (8, 8), (3, 4), (1, 2), (4, 4), (8, 3)]
    acts = [(NONE, NONE), (LEAKY, NONE), (NONE, RELU), (LEAKY, LEAKY), (RELU, NONE)]
    skips = [0, F32, 0, PLANAR, U8]
    cases = []
    i = 0
    for fi in fmts:
        for fo in fmts:
            kind = kinds[i % 4]
            ci, co = chans[i % len(chans)]
            groups = i % 3 == 1
            if groups:
                co = ci * (1 if co < ci or co % ci else co // ci)
            pre, post = acts[i % len(acts)]
            h, w = (8, 12) if kind == S2 else ((5, 7) if i % 5 == 2 and SPLIT not in (fi, fo) else (6, 10))
            cases.append(DirectCase(kind, ci, co, groups, fi, fo, R if i % 2 else Z, skips[i % 5],
                                    aux=i % 2 == 0 and fo != F32, pre=pre, post=post, h=h, w=w))
            i += 1
    # the tiled stem path (S1, c_in <= 4, c_out <= 4, dense) with every output format
    for j, fo in enumerate(fmts):
        cases.append(DirectCase(S1, 3 - j % 3, 1 + j, False, [U8, F32][j % 2], fo, [R, Z][j % 2],
                                skip=[F32, PLANAR, U8, 0][j], aux=j % 2 == 1, pre=LEAKY,
                                post=[NONE, RELU][j % 2], n=1, h=[2, 70, 18, 16][j], w=[2, 130, 66, 6][j]))
    # the general path on wider channel counts and the smallest sizes
    cases.append(DirectCase(S2, 8, 8, True, PLANAR, PLANAR, R, n=1, h=2, w=2))
    cases.append(DirectCase(T2, 4, 8, False, SPLIT, U8, Z, aux=True, n=3, h=2, w=2))
    cases.append(DirectCase(T1, 8, 1, False, PLANAR, F32, Z, skip=F32, h=7, w=5))
    for k, c in enumerate(cases):
        c.seed = 3000 + k
    return cases


DIRECT_CASES = _direct_cases()


@pytest.mark.gpu
@pytest.mark.parametrize('case', DIRECT_CASES, ids=[c.id for c in DIRECT_CASES])
def test_direct_against_float64_reference(case):
    g = _gen(case.seed)
    n, ci, co, h, w = case.n, case.c_in, case.c_out, case.h, case.w
    u8 = torch.randint(0, 256, (n, ci, h, w), generator=g, dtype=torch.uint8)
    if case.in_fmt == U8:
        x, xin = u8.float() / 255.0, u8
    else:
        x = _randn(g, n, ci, h, w)
        if case.in_fmt in (PLANAR, SPLIT):
            x = x.half().float()
        xin = x
    wt = _weights(g, case.kind, ci, co, groups=case.groups)
    b = _randn(g, co, s=0.2) + (0.4 if case.out_fmt == U8 else 0.0)
    if case.out_fmt == U8:
        wt = wt * 0.2
    oh, ow = _out_size(case.kind, h, w)
    skip = sk = None
    if case.skip:
        su8 = torch.randint(0, 256, (n, co, oh, ow), generator=g, dtype=torch.uint8)
        if case.skip == U8:
            skip, sk = su8.float() / 255.0, in_act(su8, U8)
        else:
            skip = _randn(g, n, co, oh, ow, s=0.3)
            if case.skip == PLANAR:
                skip = skip.half().float()
            sk = in_act(skip, case.skip)
    xa = in_act(xin, case.in_fmt, REFLECT if case.in_fmt in (PLANAR, SPLIT) else KEEP)
    halo = REFLECT if min(oh, ow) >= 2 else KEEP
    buf, out = out_act(case.out_fmt, n, co, oh, ow, halo)
    abuf = aux = None
    if case.aux:
        abuf, aux = guarded((n, co, oh, ow), torch.float32)
    _ops.conv(case.kind, xa, wt.cuda(), co, out, igemm=False, bias=b.cuda(), skip=sk,
              pre_act=case.pre, post_act=case.post, pad_mode=case.pad, aux=aux,
              groups=ci if case.groups else 1)
    torch.cuda.synchronize()
    pad = case.pad if not _transposed(case.kind) else Z
    ref, S, _ = ref_conv(case.kind, x, wt, b, None, case.pre, case.post, skip, pad_mode=pad,
                         groups=case.groups, path='exact')
    bound = ACC_F32 * S
    if aux is not None:
        check_close('direct', case.id + ' aux', aux.cpu(), ref, bound)
        assert guards_intact(abuf), f'{case.id}: store outside aux'
    if case.out_fmt == F32:
        check_close('direct', case.id, out.t.cpu(), ref, bound)
        assert guards_intact(buf)
    elif case.out_fmt == U8:
        u = out.t.cpu().permute(0, 3, 1, 2)
        assert guards_intact(buf)
        if aux is not None:
            assert torch.equal(u, (aux.cpu() * 255.0).clamp(0, 255).to(torch.uint8))
        check_u8('direct', case.id, u, ref, bound)
    else:
        got = unpack_layout(out.t.view(torch.int16), case.out_fmt, n, co, oh, ow).interior
        allow = bound + torch.maximum(ulp16(ref), ulp16(got.view(torch.float16)))
        # the tiled stem path writes plane 0 only (include/cae_b200.h, cae_conv_direct)
        stem = case.kind == S1 and not case.groups and ci <= 4 and co <= 4
        check_act_output('direct', case.id, buf, out, ref, allow, n, co, oh, ow, halo,
                         rel=False, padded_planes_written=not stem)


# ================================================================== layout kernels
@pytest.mark.gpu
@pytest.mark.parametrize('fmt', [PLANAR, SPLIT])
@pytest.mark.parametrize('n,c,h,w', [(1, 3, 2, 2), (2, 16, 6, 10), (1, 20, 5, 7), (3, 48, 18, 34)])
def test_layout_kernels_match_the_torch_helpers(fmt, n, c, h, w):
    if fmt == SPLIT and (h % 2 or w % 2):
        pytest.skip('split layout needs even sizes')
    g = _gen(n * 1000 + c * 10 + h)
    x = _randn(g, n, c, h, w, s=3.0)
    for halo in (KEEP, REFLECT):
        a = _ops.nchw_to_planar(x.cuda(), fmt=fmt, halo=halo)
        torch.cuda.synchronize()
        want = pack_layout(x, fmt, halo)
        assert torch.equal(a.t.cpu().view(torch.int16), want.view(torch.int16)), halo
        back = _ops.planar_to_nchw(a).cpu()
        assert torch.equal(back, x.half().float())
    if fmt == PLANAR:
        sym = torch.randint(-300, 300, (n, c, h, w), generator=g, dtype=torch.int32)
        med = torch.rand(c, generator=g) * 4 - 2
        dst = _ops.alloc_act(PLANAR, n, c, h, w)
        sym_d, med_d = sym.cuda(), med.cuda()
        C.check(C.lib().cae_eb_dequantize_planar(sym_d.data_ptr(), med_d.data_ptr(), n, c, h, w,
                                                 dst.desc(), _ops._stream_ptr(dst.t)))
        torch.cuda.synchronize()
        want = pack_layout(sym.float() + med.reshape(1, -1, 1, 1), PLANAR, KEEP)
        assert torch.equal(dst.t.cpu().view(torch.int16), want.view(torch.int16))
