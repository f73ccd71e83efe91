"""The tensor-core SR kernels (csrc/sr_tc.cu) one entry point at a time, called through the C ABI, against a float64 reference of the same
operation built from oracle/real3d_oracle.py.

Bars (error / max|reference|), per path:
  tc   fp16 operands, fp32 accumulation: the reference uses the same fp16-rounded operands; 2e-3 (the fp16 rounding of the output)
  tcx  split fp16 operands ([hi | lo], `sr_mode='tc_exact'`): the reference uses the UNROUNDED fp32 operands and outputs are read back as
       hi + lo; 1e-5 - about 30x below what fp16 operands give (3e-4) and far below a dropped cross term (~2^-11)
  fused ToRGB images are compared against the float64 activation before any fp16 rounding, since the epilogue reads the fp32 value.
Elementwise kernels compute in fp32 and are compared with the same formula in torch fp32 (within an ulp or two of the output type).
The persistent cases launch more work units than the GPU has SMs, so the unit loop, the parity wrap of the double-buffered accumulators and
the strip / tap ring wraps across units all run; each asserts that it still does.

Run as a script (`python tests/test_gpu_sr_kernels.py OUT.pt`) it writes the GPU outputs of the variant cases to OUT.pt: the kernel variants
selected by R3DP_TC_ROWS / R3DP_TC_MIX are read once per process, so test_env_kernel_variants_are_bit_identical runs them in a child."""
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import pytest  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from oracle import real3d_oracle as orc  # noqa: E402
from real3dportrait_b200 import _capi as capi  # noqa: E402
from real3dportrait_b200 import sr_tc  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = 'cuda'
H16 = torch.float16
TC_BAR, TCX_BAR = 2e-3, 1e-5
#: standard deviation of every activation fed to the conv kernels; the split path is fp32-grade only from 2^-4 up (test_cpu_split_conv.py)
ACT_SCALE = 1.0
R_DEFAULT = 2                 # output rows per conv tile unless R3DP_TC_ROWS says otherwise
VARIANT_ENV = ('R3DP_TC_ROWS', 'R3DP_TC_MIX')


def _pad64(c):
    return (c + 63) // 64 * 64


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _units(N, phases, rows, W, R=R_DEFAULT):
    """Work units of one conv_tc3 launch (launch_conv3_rs): row groups padded so a CTA pair shares (image, phase)."""
    rg, tiles = -(-rows // R), W // 128
    if (rg * tiles) & 1:
        rg += 1
    return N * phases * rg * tiles


def _report(name, got, ref, bar, scale=None):
    scale = float(ref.abs().max()) if scale is None else scale
    err = float((got.double() - ref.double()).abs().max()) / scale
    print(f'{name}: max|err| / max|ref| = {err:.2e} (bar {bar:.0e}, max|ref| {scale:.3g})')
    assert err < bar, (name, err, bar)
    return err


def _ulp16(v):
    """Spacing of fp16 numbers at |v| (subnormal spacing below 2^-14)."""
    a = v.double().abs().clamp_min(2.0 ** -14)
    return torch.exp2(torch.floor(torch.log2(a)) - 10)


def _weights(g, Nw, O, I, k=3):
    w = torch.randn(Nw, O, I, k, k, generator=g)
    return w / w.square().sum(dim=(2, 3, 4), keepdim=True).sqrt()            # demodulated: unit-norm filters, as fold_weight leaves them


def _act_nhwc(x, split):
    """fp32 NCHW [N,C,H,W] -> NHWC fp16 [N,H,W,Cp] (zero padded), or the split layout [N,H,W,2*Cp] = [hi | lo] with lo = fp16(x - hi)."""
    N, C, H, W = x.shape
    Cp = _pad64(C)
    xn = x.permute(0, 2, 3, 1)
    hi = xn.half()
    out = torch.zeros(N, H, W, Cp * (2 if split else 1), dtype=H16)
    out[..., :C] = hi
    if split:
        out[..., Cp:Cp + C] = (xn - hi.float()).half()
    return out.to(DEV)


def _from_nhwc(y, C, split):
    """NHWC fp16 output -> float64 NCHW [N,C,H,W]; split outputs are read back as hi + lo (lo starts C channels after hi)."""
    y = y.cpu().double()
    v = y[..., :C] + (y[..., C:2 * C] if split else 0)
    return v.permute(0, 3, 1, 2)


def _operands(x, wf, split):
    """Reference operands: the fp16-rounded ones the tc kernel multiplies, or the unrounded fp32 ones the tcx kernel represents."""
    if split:
        return x.double(), wf.double()
    return x.half().double(), wf.half().double()


def _per_sample(wf, N):
    return wf.expand(N, *wf.shape[1:]) if wf.shape[0] == 1 else wf


def _pack(wf, split, composed=False):
    Nw, O, I = wf.shape[:3]
    wd = wf.to(DEV)
    out = torch.empty(Nw, 36 if composed else 9, O, _pad64(I) * (2 if split else 1), device=DEV, dtype=H16)
    name = 'pack_weights_up_composed' if composed else 'pack_weights'
    capi.check(sr_tc._fn(name, split)(capi.ptr(wd), Nw, O, I, capi.ptr(out, H16), capi.stream()))
    return out


# ---------------------------------------------------------------------------------------------------------------------------------------------
# SynthesisLayer convolutions: r3dp_sr_tc(x)_layer (up 1 and the two-step up 2) and r3dp_sr_tc(x)_layer_up_composed
# ---------------------------------------------------------------------------------------------------------------------------------------------
#: id -> (up, composed, N, Nw, I, O, H, W, persistent)
LAYER_CASES = {
    'up1_H5': (1, False, 2, 2, 64, 128, 5, 128, False),          # 3 row groups, padded to 4
    'up1_I96': (1, False, 2, 2, 96, 128, 4, 128, False),         # I not a multiple of 64
    'up1_N3_Nw1': (1, False, 3, 1, 64, 128, 4, 128, False),      # shared weights
    'up1_N3_Nw3': (1, False, 3, 3, 64, 128, 4, 128, False),      # per-sample weights
    'up1_O256': (1, False, 2, 2, 64, 256, 4, 128, False),        # two cout blocks per unit
    'up1_persistent': (1, False, 3, 3, 64, 256, 64, 256, True),
    'up2_H5': (2, False, 2, 2, 128, 128, 5, 128, False),         # phase rows H+1 (even output rows) vs H
    'up2_W256': (2, False, 2, 2, 128, 128, 4, 256, False),       # even x-block count: phases interleaved
    'up2_I256': (2, False, 2, 1, 256, 128, 4, 128, False),
    'up2_persistent': (2, False, 2, 2, 128, 128, 64, 256, True),
    'upc_I7': (2, True, 2, 2, 7, 128, 4, 128, False),
    'upc_I32': (2, True, 2, 1, 32, 256, 5, 128, False),
    'upc_persistent': (2, True, 2, 2, 32, 256, 32, 256, True),
}
#: fp16 cases that test_gpu_parity.py::test_tc_layer_vs_oracle covers (its N = 2 parametrization); here they run split only
TC_IN_PARITY = {'up1_H5', 'up1_I96', 'up1_O256', 'up2_H5', 'up2_W256', 'up2_I256'}


def _layer_inputs(case, seed):
    up, composed, N, Nw, I, O, H, W, _ = LAYER_CASES[case]
    g = torch.Generator().manual_seed(seed)
    return ACT_SCALE * torch.randn(N, I, H, W, generator=g), _weights(g, Nw, O, I), 0.1 * torch.randn(O, generator=g)


def _run_layer(case, split, x, wf, bias):
    up, composed, N, Nw, I, O, H, W, _ = LAYER_CASES[case]
    xin, wp, b = _act_nhwc(x, split), _pack(wf, split, composed), bias.to(DEV)
    wide = 2 if split else 1
    y = torch.empty(N, H * up, W * up, O * wide, device=DEV, dtype=H16)
    if composed:
        capi.check(sr_tc._fn('layer_up_composed', split)(capi.ptr(xin, H16), capi.ptr(wp, H16), capi.ptr(b), N, Nw, I, O, H, W, capi.ptr(y, H16),
                                                          capi.stream()))
    else:
        scratch = torch.empty(sr_tc._fn('scratch_bytes', split)(N, O, H, W), device=DEV, dtype=torch.uint8) if up == 2 else None
        capi.check(sr_tc._fn('layer', split)(capi.ptr(xin, H16), capi.ptr(wp, H16), capi.ptr(b), N, Nw, I, O, H, W, up, capi.ptr(y, H16),
                                             capi.ptr(scratch, torch.uint8), capi.stream()))
    torch.cuda.synchronize()
    return y


def _layer_ref(case, split, x, wf, bias):
    up, _, N = LAYER_CASES[case][:3]
    xr, wr = _operands(x, wf, split)
    return orc.lrelu_gain(orc.mod_conv(xr, _per_sample(wr, N), up), bias.double())


@pytest.mark.parametrize('case,split', [(c, s) for c in LAYER_CASES for s in (False, True) if s or c not in TC_IN_PARITY])
def test_layer_vs_float64(case, split):
    up, composed, N, Nw, I, O, H, W, persistent = LAYER_CASES[case]
    if persistent:
        units = _units(N, 4 if up == 2 else 1, H + 1 if (up == 2 and not composed) else H, W)
        assert units > _sms(), (units, _sms())
    x, wf, bias = _layer_inputs(case, seed=11)
    y = _run_layer(case, split, x, wf, bias)
    ref = _layer_ref(case, split, x, wf, bias)
    got = _from_nhwc(y, O, split)
    assert got.shape == ref.shape
    _report(f'layer {case} {"tcx" if split else "tc"}', got, ref, TCX_BAR if split else TC_BAR)


# ---------------------------------------------------------------------------------------------------------------------------------------------
# fused ToRGB epilogues
# ---------------------------------------------------------------------------------------------------------------------------------------------
def _rgb_ref(act, wrgb, brgb, img_prev, same_res=False):
    """ToRGB (1x1 conv of the fp32 activation) + bias + skip image (FIR-upsampled, or as is at the same resolution)."""
    y = torch.einsum('nchw,nkc->nkhw', act, _per_sample(wrgb.double(), act.shape[0])) + brgb.double().view(1, 3, 1, 1)
    if img_prev is not None:
        y = y + (img_prev.double() if same_res else orc.upsample2x(img_prev.double()))
    return y


def _torgb_inputs(g, N, Nw, O, H, W, same_res, rgb_gain=1.0):
    wrgb = rgb_gain * torch.randn(Nw, 3, O, generator=g) / math.sqrt(O)
    brgb = 0.1 * torch.randn(3, generator=g)
    img_prev = 0.5 * torch.randn(N, 3, H if same_res else H // 2, W if same_res else W // 2, generator=g)
    return wrgb, brgb, img_prev


def _run_layer_torgb(split, N, Nw, I, O, H, W, x, wf, bias, wrgb, brgb, img_prev, noup=False):
    xin, wp = _act_nhwc(x, split), _pack(wf, split)
    b, wr, br, ip = bias.to(DEV), wrgb.to(DEV), brgb.to(DEV), img_prev.to(DEV)
    y = torch.empty(N, H, W, O * (2 if split else 1), device=DEV, dtype=H16)
    img = torch.empty(N, 3, H, W, device=DEV)
    fn = capi.lib().r3dp_sr_tc_layer_torgb_noup if noup else sr_tc._fn('layer_torgb', split)
    capi.check(fn(capi.ptr(xin, H16), capi.ptr(wp, H16), capi.ptr(b), capi.ptr(wr), capi.ptr(br), capi.ptr(ip), N, Nw, I, O, H, W,
                  capi.ptr(y, H16), capi.ptr(img), capi.stream()))
    torch.cuda.synchronize()
    return y, img


def _torgb_case(seed, N, Nw, I, O, H, W, same_res):
    g = torch.Generator().manual_seed(seed)
    x, wf, bias = ACT_SCALE * torch.randn(N, I, H, W, generator=g), _weights(g, Nw, O, I), 0.1 * torch.randn(O, generator=g)
    return (x, wf, bias) + _torgb_inputs(g, N, Nw, O, H, W, same_res)


@pytest.mark.parametrize('split', [False, True], ids=['tc', 'tcx'])
@pytest.mark.parametrize('O,shared', [(128, False), (128, True), (256, False), (256, True)])
def test_layer_torgb_vs_float64(split, O, shared):
    N, I, H, W = 2, 64, 6, 128
    Nw = 1 if shared else N
    x, wf, bias, wrgb, brgb, img_prev = _torgb_case(21, N, Nw, I, O, H, W, False)
    y, img = _run_layer_torgb(split, N, Nw, I, O, H, W, x, wf, bias, wrgb, brgb, img_prev)
    xr, wr = _operands(x, wf, split)
    act = orc.lrelu_gain(orc.mod_conv(xr, _per_sample(wr, N), 1), bias.double())
    bar = TCX_BAR if split else TC_BAR
    tag = f'layer_torgb {"tcx" if split else "tc"} O={O} Nw={Nw}'
    _report(tag + ' y', _from_nhwc(y, O, split), act, bar)
    _report(tag + ' img', img.cpu(), _rgb_ref(act, wrgb, brgb, img_prev), bar)


@pytest.mark.parametrize('O,shared', [(128, False), (256, True)])
def test_layer_torgb_noup_vs_float64(O, shared):
    """SynthesisBlockNoUp tail: the skip image has the OUTPUT resolution and is added as is.  H = 5: this entry point takes odd heights."""
    N, I, H, W = 2, 64, 5, 128
    Nw = 1 if shared else N
    x, wf, bias, wrgb, brgb, img_prev = _torgb_case(22, N, Nw, I, O, H, W, True)
    y, img = _run_layer_torgb(False, N, Nw, I, O, H, W, x, wf, bias, wrgb, brgb, img_prev, noup=True)
    xr, wr = _operands(x, wf, False)
    act = orc.lrelu_gain(orc.mod_conv(xr, _per_sample(wr, N), 1), bias.double())
    _report(f'layer_torgb_noup O={O} Nw={Nw} y', _from_nhwc(y, O, False), act, TC_BAR)
    _report(f'layer_torgb_noup O={O} Nw={Nw} img', img.cpu(), _rgb_ref(act, wrgb, brgb, img_prev, same_res=True), TC_BAR)


@pytest.mark.parametrize('same_res', [0, 1])
def test_torgb_ex_vs_float64(same_res):
    N, C, H, W = 2, 136, 6, 10
    g = torch.Generator().manual_seed(23 + same_res)
    x16 = (ACT_SCALE * torch.randn(N, H, W, C, generator=g)).half()
    wrgb, brgb, img_prev = _torgb_inputs(g, N, N, C, H, W, same_res)
    xd, wr, br, ip = x16.to(DEV), wrgb.to(DEV), brgb.to(DEV), img_prev.to(DEV)
    img = torch.empty(N, 3, H, W, device=DEV)
    capi.check(capi.lib().r3dp_sr_tc_torgb_ex(capi.ptr(xd, H16), capi.ptr(wr), capi.ptr(br), capi.ptr(ip), same_res, N, N, C, H, W, capi.ptr(img),
                                              capi.stream()))
    torch.cuda.synchronize()
    ref = _rgb_ref(x16.double().permute(0, 3, 1, 2), wrgb, brgb, img_prev, same_res=bool(same_res))
    _report(f'torgb_ex same_res={same_res}', img.cpu(), ref, TCX_BAR)          # fp32 dot products of fp16 inputs


@pytest.mark.parametrize('split', [False, True], ids=['tc', 'tcx'])
@pytest.mark.parametrize('mode', ['f32', 'clamp', 'u8'])
def test_last_layer_vs_float64(split, mode):
    """last conv (I -> 128) fused with ToRGB + skip; clamp to [-1, 1]; uint8 HWC frames = int((clamp(x) + 1) / 2 * 255).  The image is scaled
    to leave [-1, 1] on both sides so the clamp acts."""
    N, I, O, H, W = 2, 64, 128, 6, 128
    Nw = N if mode == 'f32' else 1
    g = torch.Generator().manual_seed(24)
    x, wf, bias = ACT_SCALE * torch.randn(N, I, H, W, generator=g), _weights(g, Nw, O, I), 0.1 * torch.randn(O, generator=g)
    wrgb, brgb, img_prev = _torgb_inputs(g, N, Nw, O, H, W, False, rgb_gain=2.0)
    xin, wp = _act_nhwc(x, split), _pack(wf, split)
    b, wr, br, ip = bias.to(DEV), wrgb.to(DEV), brgb.to(DEV), img_prev.to(DEV)
    img = torch.empty(N, 3, H, W, device=DEV)
    u8 = torch.empty(N, H, W, 3, device=DEV, dtype=torch.uint8)
    fn = capi.lib().r3dp_sr_tcx_last_layer if split else capi.lib().r3dp_sr_tc_last_layer_ex
    capi.check(fn(capi.ptr(xin, H16), capi.ptr(wp, H16), capi.ptr(b), capi.ptr(wr), capi.ptr(br), capi.ptr(ip), N, Nw, I, H, W,
                  None if mode == 'u8' else capi.ptr(img), capi.ptr(u8, torch.uint8) if mode == 'u8' else None, int(mode == 'clamp'), capi.stream()))
    torch.cuda.synchronize()
    xr, wrf = _operands(x, wf, split)
    ref = _rgb_ref(orc.lrelu_gain(orc.mod_conv(xr, _per_sample(wrf, N), 1), bias.double()), wrgb, brgb, img_prev)
    assert (ref > 1).any() and (ref < -1).any() and (ref.abs() < 1).any()
    bar = TCX_BAR if split else TC_BAR
    tag = f'last_layer {"tcx" if split else "tc"} {mode}'
    scale = float(ref.abs().max())                      # the error scales with the image BEFORE the (1-Lipschitz) clamp
    if mode != 'u8':
        _report(tag, img.cpu(), ref.clamp(-1, 1) if mode == 'clamp' else ref, bar, scale)
        return
    tol = bar * scale

    def frame(v):
        return ((v.clamp(-1, 1) + 1) / 2 * 255).floor()
    want, lo, hi = frame(ref), frame(ref - tol), frame(ref + tol)
    near = lo != hi                         # the float64 value lies within the error bar of a quantisation boundary
    got = u8.cpu().permute(0, 3, 1, 2).double()
    print(f'{tag}: {int(near.sum())} of {near.numel()} values within the error bar of a quantisation boundary')
    assert torch.equal(got[~near], want[~near])
    assert bool(((got[near] >= lo[near]) & (got[near] <= hi[near])).all())


# ---------------------------------------------------------------------------------------------------------------------------------------------
# plain convolutions of the torso head / large_sr: r3dp_sr_tc_conv_res and r3dp_sr_tcx_conv
# ---------------------------------------------------------------------------------------------------------------------------------------------
def _act_ref(v, act):
    if act == 0:
        return v
    if act == 1:
        return F.leaky_relu(v, 0.2) * math.sqrt(2.0)
    if act == 2:
        return F.leaky_relu(v, 0.01)
    return F.relu(v)


def _plain_conv(seed, I, Oc, k):
    torch.manual_seed(seed)
    conv = torch.nn.Conv2d(I, Oc, k, padding=k // 2)
    with torch.no_grad():
        conv.bias.copy_(0.1 * torch.randn(Oc))
    return conv


@pytest.mark.parametrize('split,ksize,act,residual', [(False, k, a, r) for k in (1, 3) for a in range(4) for r in (False, True)] +
                         [(True, k, a, False) for k in (1, 3) for a in range(4)])
def test_conv_vs_float64(split, ksize, act, residual):
    """nn.Conv2d (+ act: 0 linear, 1 lrelu(0.2)*sqrt2, 2 nn.LeakyReLU(0.01), 3 ReLU) [+ residual added after the activation, ResBlock2d].  100
    output channels are padded to 128 by pack_plain's zero filters; I = 96 pads the input to 128."""
    N, I, Oc, H, W = 2, 96, 100, 4, 128
    conv = _plain_conv(31 + ksize, I, Oc, ksize)
    g = torch.Generator().manual_seed(32 + act)
    x = ACT_SCALE * torch.randn(N, I, H, W, generator=g)
    wp, bias, k = sr_tc.pack_plain(conv.to(DEV), I, split=split)
    O = wp.shape[2]
    xin = _act_nhwc(x, split)
    y = torch.empty(N, H, W, O * (2 if split else 1), device=DEV, dtype=H16)
    res = (ACT_SCALE * torch.randn(N, H, W, O, generator=g)).half() if residual else None
    rd = res.to(DEV) if residual else None
    if split:
        capi.check(capi.lib().r3dp_sr_tcx_conv(capi.ptr(xin, H16), capi.ptr(wp, H16), capi.ptr(bias), N, 1, I, O, H, W, k, act, capi.ptr(y, H16),
                                               capi.stream()))
    else:
        capi.check(capi.lib().r3dp_sr_tc_conv_res(capi.ptr(xin, H16), capi.ptr(wp, H16), capi.ptr(bias), N, 1, I, O, H, W, k, act,
                                                  capi.ptr(rd, H16), capi.ptr(y, H16), capi.stream()))
    torch.cuda.synchronize()
    w = torch.zeros(O, I, ksize, ksize)
    w[:Oc] = conv.weight.detach().cpu()
    b = torch.zeros(O, dtype=torch.float64)
    b[:Oc] = conv.bias.detach().cpu().double()
    xr, wr = _operands(x, w, split)
    ref = _act_ref(F.conv2d(xr, wr, b, padding=ksize // 2), act)
    if residual:
        ref = ref + res.double().permute(0, 3, 1, 2)
    _report(f'conv {"tcx" if split else "tc"} k={ksize} act={act}{" +res" if residual else ""}', _from_nhwc(y, O, split), ref,
            TCX_BAR if split else TC_BAR)


# ---------------------------------------------------------------------------------------------------------------------------------------------
# elementwise kernels (fp32 arithmetic): the same formula in torch fp32
# ---------------------------------------------------------------------------------------------------------------------------------------------
def _max_ulp16(got, ref32):
    return float(((got.double() - ref32.double()).abs() / _ulp16(ref32)).max())


@pytest.mark.parametrize('xb_shared', [0, 1])
def test_alpha_cat_ex(xb_shared):
    N, H, W, Ca, sa, Cb, sb = 2, 5, 12, 48, 64, 24, 40                        # pixel strides larger than the channel counts
    g = torch.Generator().manual_seed(41)
    xa = torch.randn(N, H, W, sa, generator=g).half()
    xb = torch.randn(1 if xb_shared else N, H, W, sb, generator=g).half()
    alpha = torch.rand(N, H, W, generator=g)
    xad, xbd, ad = xa.to(DEV), xb.to(DEV), alpha.to(DEV)
    out = torch.empty(N, H, W, Ca + Cb, device=DEV, dtype=H16)
    capi.check(capi.lib().r3dp_sr_alpha_cat_ex(capi.ptr(xad, H16), Ca, sa, capi.ptr(xbd, H16), Cb, sb, xb_shared, capi.ptr(ad), N, H, W,
                                               capi.ptr(out, H16), capi.stream()))
    torch.cuda.synchronize()
    al = alpha[..., None]
    ref = torch.cat([xa[..., :Ca].float() * al, xb[..., :Cb].float().expand(N, -1, -1, -1) * (1 - al)], dim=-1)
    e = _max_ulp16(out.cpu(), ref)
    print(f'alpha_cat_ex xb_shared={xb_shared}: {e:.2f} fp16 ulp')
    assert e <= 1.0


def test_alpha_mix():
    N, H, W, C, sa, sb = 2, 5, 12, 40, 48, 64
    g = torch.Generator().manual_seed(42)
    xa, xb = torch.randn(N, H, W, sa, generator=g).half(), torch.randn(N, H, W, sb, generator=g).half()
    alpha = torch.rand(N, H, W, generator=g)
    xad, xbd, ad = xa.to(DEV), xb.to(DEV), alpha.to(DEV)
    out = torch.empty(N, H, W, C, device=DEV, dtype=H16)
    capi.check(capi.lib().r3dp_sr_alpha_mix(capi.ptr(xad, H16), sa, capi.ptr(xbd, H16), sb, capi.ptr(ad), C, N, H, W, capi.ptr(out, H16),
                                            capi.stream()))
    torch.cuda.synchronize()
    al = alpha[..., None]
    ref = xa[..., :C].float() * al + xb[..., :C].float() * (1 - al)
    e = _max_ulp16(out.cpu(), ref)
    print(f'alpha_mix: {e:.2f} fp16 ulp')
    assert e <= 1.0


def _gate(y, stride, lo_off, cap, N, H, W):
    out = torch.empty(N, 1, H, W, device=DEV)
    capi.check(capi.lib().r3dp_sr_alpha_gate(capi.ptr(y, H16), stride, lo_off, capi.ptr(cap), N, H, W, capi.ptr(out), capi.stream()))
    torch.cuda.synchronize()
    return out.cpu()


def _assert_f32_close(name, got, ref, scale, ulps=4):
    """|got - ref| within `ulps` fp32 ulps of `scale` (the magnitude the rounding errors scale with)."""
    e = float(((got.double() - ref.double()).abs() / (scale.double() * torch.finfo(torch.float32).eps).clamp_min(1e-45)).max())
    print(f'{name}: {e:.2f} fp32 ulp')
    assert e <= ulps, (name, e)


def test_alpha_gate_lo_off_zero():
    N, H, W, stride = 2, 6, 20, 8
    g = torch.Generator().manual_seed(43)
    y = (3 * torch.randn(N, H, W, stride, generator=g)).half()
    cap = torch.rand(N, 1, H, W, generator=g)
    yd, cd = y.to(DEV), cap.to(DEV)
    got = _gate(yd, stride, 0, cd, N, H, W)
    ref = torch.minimum(torch.sigmoid(y[..., 0].float()).view(N, 1, H, W), cap)
    _assert_f32_close('alpha_gate lo_off=0', got, ref, ref.abs())


def test_alpha_gate_on_split_conv_output():
    """fuse mode v3: the logit is the split output of r3dp_sr_tcx_conv (channel 0 + its lo half lo_off channels further)."""
    N, I, H, W = 2, 32, 4, 128
    conv = _plain_conv(44, I, 1, 3)
    g = torch.Generator().manual_seed(45)
    x = ACT_SCALE * torch.randn(N, I, H, W, generator=g)
    cap = 0.5 + 0.5 * torch.rand(N, 1, H, W, generator=g)
    wp, bias, k = sr_tc.pack_plain(conv.to(DEV), I, split=True)
    O = wp.shape[2]
    xin = _act_nhwc(x, True)
    y = torch.empty(N, H, W, 2 * O, device=DEV, dtype=H16)
    capi.check(capi.lib().r3dp_sr_tcx_conv(capi.ptr(xin, H16), capi.ptr(wp, H16), capi.ptr(bias), N, 1, I, O, H, W, k, 0, capi.ptr(y, H16),
                                           capi.stream()))
    cd = cap.to(DEV)
    got, hi_only = _gate(y, 2 * O, O, cd, N, H, W), _gate(y, 2 * O, 0, cd, N, H, W)
    yc = y.cpu()
    logit32 = (yc[..., 0].float() + yc[..., O].float()).view(N, 1, H, W)
    ref32 = torch.minimum(torch.sigmoid(logit32), cap)
    _assert_f32_close('alpha_gate lo_off>0', got, ref32, ref32.abs())
    assert not torch.equal(got, hi_only)                                      # the lo half is read
    # against float64: sigmoid is 0.25-Lipschitz, so the split conv's bar on the logit carries over scaled by 0.25 (+ fp32 sigmoid rounding)
    logit64 = F.conv2d(x.double(), conv.weight.detach().cpu().double(), conv.bias.detach().cpu().double(), padding=1)
    ref64 = torch.minimum(torch.sigmoid(logit64), cap.double())
    err, bound = float((got.double() - ref64).abs().max()), 0.25 * TCX_BAR * float(logit64.abs().max()) + 1e-6
    print(f'alpha_gate on tcx_conv vs float64: max|err| {err:.2e} (bound {bound:.1e})')
    assert err < bound


def test_blend():
    N, C, H, W = 2, 3, 7, 33
    g = torch.Generator().manual_seed(46)
    a, b = torch.randn(N, C, H, W, generator=g), torch.randn(N, C, H, W, generator=g)
    alpha = torch.rand(N, 1, H, W, generator=g)
    ad, bd, al = a.to(DEV), b.to(DEV), alpha.to(DEV)
    out = torch.empty(N, C, H, W, device=DEV)
    capi.check(capi.lib().r3dp_sr_blend(capi.ptr(ad), capi.ptr(bd), capi.ptr(al), N, C, H, W, capi.ptr(out), capi.stream()))
    torch.cuda.synchronize()
    ref = a * alpha + b * (1 - alpha)
    _assert_f32_close('blend', out.cpu(), ref, (a * alpha).abs() + (b * (1 - alpha)).abs(), ulps=2)


def test_person_occlusion_threshold_is_strict():
    """clamp(torso + (head > thr ? 1 : head), 0, 1): `>` as in the reference (sr_with_ref.py:118), so head == thr keeps head, it does not
    become 1."""
    N, H, W, thr = 2, 8, 16, 0.9
    g = torch.Generator().manual_seed(47)
    head = torch.rand(N, H, W, generator=g)
    head.view(-1)[::5] = torch.tensor(thr, dtype=torch.float32)              # exactly at the threshold (the same fp32 value the C call gets)
    torso = 1.2 * torch.rand(N, H, W, generator=g) - 0.3
    hd, td = head.to(DEV), torso.to(DEV)
    out = torch.empty(N, H, W, device=DEV)
    capi.check(capi.lib().r3dp_sr_person_occlusion(capi.ptr(hd), capi.ptr(td), thr, N, H, W, capi.ptr(out), capi.stream()))
    torch.cuda.synchronize()
    got = out.cpu()
    t32 = torch.tensor(thr, dtype=torch.float32)
    ref = (torso + torch.where(head > t32, torch.ones_like(head), head)).clamp(0, 1)
    eq = head == t32
    assert eq.any() and (head > t32).any() and ((torso + head) > 1).any() and ((torso + head) < 0).any()
    assert torch.equal(got, ref)
    assert torch.equal(got[eq], (torso[eq] + t32).clamp(0, 1))
    assert not torch.equal(got[eq], (torso[eq] + 1).clamp(0, 1))


# ---------------------------------------------------------------------------------------------------------------------------------------------
# input kernels: bilinear (align_corners=False) resize to NHWC fp16 [| lo], channels padded with zeros
# ---------------------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('split', [0, 1], ids=['tc', 'tcx'])
@pytest.mark.parametrize('copy', [False, True], ids=['resize', 'copy'])
@pytest.mark.parametrize('kind', ['nchw', 'nhwc', 'nhwc_rgb'])
def test_input_kernels(kind, copy, split):
    N, size = 2, 128 if not copy else 64
    C = 35 if kind == 'nchw' else 40                                         # NHWC sources need C % 8 == 0
    h, w = (64, 64) if copy else (48, 40)                                     # resize ratios 8/3 and 16/5
    g = torch.Generator().manual_seed(51)
    x = ACT_SCALE * torch.randn(N, C, h, w, generator=g)                       # logical NCHW image
    Cp = _pad64(C)
    y = torch.empty(N, size, size, Cp * (2 if split else 1), device=DEV, dtype=H16)
    rgb = torch.empty(N, 3, size, size, device=DEV)
    L = capi.lib()
    if kind == 'nchw':
        src = x.to(DEV)
        capi.check((L.r3dp_sr_tcx_input if split else L.r3dp_sr_tc_input)(capi.ptr(src), N, C, h, w, size, capi.ptr(y, H16), capi.stream()))
    else:
        src = x.permute(0, 2, 3, 1).contiguous().to(DEV)
        if kind == 'nhwc':
            capi.check((L.r3dp_sr_tcx_input_nhwc if split else L.r3dp_sr_tc_input_nhwc)(capi.ptr(src), N, C, h, w, size, capi.ptr(y, H16),
                                                                                      capi.stream()))
        else:
            capi.check(L.r3dp_sr_tc_input_nhwc_rgb(capi.ptr(src), N, C, h, w, size, capi.ptr(y, H16), capi.ptr(rgb), split, capi.stream()))
    torch.cuda.synchronize()
    yc = y.cpu()
    hi = yc[..., :C]
    assert not yc[..., C:Cp].any()                                            # pad channels exactly zero
    if split:
        assert not yc[..., Cp + C:].any()
    tag = f'input {kind} {"tcx" if split else "tc"} {"copy" if copy else "resize"}'
    if copy:
        xn = x.permute(0, 2, 3, 1)
        assert torch.equal(hi, xn.half())
        if split:
            assert torch.equal(yc[..., Cp:Cp + C], (xn - xn.half().float()).half())
        if kind == 'nhwc_rgb':
            assert torch.equal(rgb.cpu(), x[:, :3])
        return
    ref = F.interpolate(x.double(), size=(size, size), mode='bilinear', align_corners=False).permute(0, 2, 3, 1)
    slack = TCX_BAR * float(ref.abs().max())                                  # fp32 source coordinates and weights
    if split:
        _report(tag, hi.double() + yc[..., Cp:Cp + C].double(), ref, TCX_BAR)
    else:
        e = float(((hi.double() - ref).abs() / (_ulp16(ref) + slack)).max())
        print(f'{tag}: {e:.2f} x (1 fp16 ulp + {slack:.1e})')
        assert e <= 1.0
    if kind == 'nhwc_rgb':
        _report(tag + ' rgb_out', rgb.cpu().double(), ref[..., :3].permute(0, 3, 1, 2), TCX_BAR)


# ---------------------------------------------------------------------------------------------------------------------------------------------
# kernel variants selected by environment variables (read once per process): R3DP_TC_ROWS = 1 | 4 output rows per tile (4: a single TMEM
# accumulator and 7 strip slots), R3DP_TC_MIX = 0 (phases not interleaved).  The K order of every output pixel - chunk, tap, k step - does not
# depend on the rows per tile or on the unit order, so the outputs must be bit-identical to the default variant's.
# ---------------------------------------------------------------------------------------------------------------------------------------------
def _variant_outputs():
    out = {}
    for split in (False, True):
        s = 'tcx' if split else 'tc'
        for case in ('up1_persistent', 'up2_persistent'):
            out[f'{case} {s}'] = _run_layer(case, split, *_layer_inputs(case, seed=61)).cpu()
        N, Nw, I, O, H, W = 2, 1, 64, 256, 6, 128
        y, img = _run_layer_torgb(split, N, Nw, I, O, H, W, *_torgb_case(62, N, Nw, I, O, H, W, False))
        out[f'layer_torgb {s} y'], out[f'layer_torgb {s} img'] = y.cpu(), img.cpu()
    return out


_default_outputs = {}


@pytest.mark.parametrize('env', [{'R3DP_TC_ROWS': '1'}, {'R3DP_TC_ROWS': '4'}, {'R3DP_TC_MIX': '0'}], ids=['rows1', 'rows4', 'mix0'])
def test_env_kernel_variants_are_bit_identical(env, tmp_path):
    base_env = {k: v for k, v in os.environ.items() if k not in VARIANT_ENV}
    if not _default_outputs:
        if any(k in os.environ for k in VARIANT_ENV):                         # this process runs a variant itself: get the default from a child
            path = tmp_path / 'default.pt'
            subprocess.run([sys.executable, os.path.abspath(__file__), str(path)], env=base_env, cwd=ROOT, timeout=600, check=True)
            _default_outputs.update(torch.load(path))
        else:
            _default_outputs.update(_variant_outputs())
    path = tmp_path / 'variant.pt'
    r = subprocess.run([sys.executable, os.path.abspath(__file__), str(path)], env=dict(base_env, **env), cwd=ROOT, timeout=600,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout[-4000:]
    got = torch.load(path)
    assert got.keys() == _default_outputs.keys()
    for k, v in _default_outputs.items():
        assert torch.equal(got[k], v), (env, k, float((got[k].double() - v.double()).abs().max()))


# ---------------------------------------------------------------------------------------------------------------------------------------------
# argument checks: a call that breaks a stated restriction returns non-zero, names the restriction, and enqueues nothing.  Buffers are sized
# for the shape passed, so a call that wrongly went ahead would still stay inside them.
# ---------------------------------------------------------------------------------------------------------------------------------------------
def _expect_rejected(call, needle):
    L = capi.lib()
    torch.cuda.synchronize()
    before = L.r3dp_launch_count()
    rc = call()
    torch.cuda.synchronize()
    msg = L.r3dp_last_error().decode()
    assert rc != 0, needle
    assert needle in msg, (needle, msg)
    assert L.r3dp_launch_count() == before, ('launched before rejecting', msg)


def _layer_call(split=False, N=2, Nw=2, I=64, O=128, H=4, W=128, up=1):
    Ip, wide = _pad64(I), (2 if split else 1)
    x = torch.zeros(N, H, W, Ip * wide, device=DEV, dtype=H16)
    wp = torch.zeros(max(Nw, 1), 9, O, Ip * wide, device=DEV, dtype=H16)
    b = torch.zeros(O, device=DEV)
    y = torch.zeros(N, H * max(up, 1), W * max(up, 1), O * wide, device=DEV, dtype=H16)
    scratch = torch.zeros(max(sr_tc._fn('scratch_bytes', split)(N, O, H, W), 1), device=DEV, dtype=torch.uint8)
    fn = sr_tc._fn('layer', split)
    return lambda: fn(capi.ptr(x, H16), capi.ptr(wp, H16), capi.ptr(b), N, Nw, I, O, H, W, up, capi.ptr(y, H16), capi.ptr(scratch, torch.uint8),
                      capi.stream())


def _fused_call(kind, split=False, N=2, Nw=2, I=64, O=128, H=4, W=128):
    Ip, wide = _pad64(I), (2 if split else 1)
    x = torch.zeros(N, H, W, Ip * wide, device=DEV, dtype=H16)
    wp = torch.zeros(Nw, 9, O, Ip * wide, device=DEV, dtype=H16)
    b, wrgb, brgb = torch.zeros(O, device=DEV), torch.zeros(Nw, 3, O, device=DEV), torch.zeros(3, device=DEV)
    prev = torch.zeros(N, 3, max(H // 2, 1), W // 2, device=DEV)
    y = torch.zeros(N, H, W, O * wide, device=DEV, dtype=H16)
    img = torch.zeros(N, 3, H, W, device=DEV)
    L, P = capi.lib(), capi.ptr
    if kind == 'layer_torgb':
        fn = sr_tc._fn('layer_torgb', split)
        return lambda: fn(P(x, H16), P(wp, H16), P(b), P(wrgb), P(brgb), P(prev), N, Nw, I, O, H, W, P(y, H16), P(img), capi.stream())
    fn = L.r3dp_sr_tcx_last_layer if split else L.r3dp_sr_tc_last_layer_ex
    return lambda: fn(P(x, H16), P(wp, H16), P(b), P(wrgb), P(brgb), P(prev), N, Nw, I, H, W, P(img), None, 0, capi.stream())


def _conv_call(split=False, ksize=3, act=0, N=2, I=64, O=128, H=4, W=128):
    Ip, wide = _pad64(I), (2 if split else 1)
    x = torch.zeros(N, H, W, Ip * wide, device=DEV, dtype=H16)
    wp = torch.zeros(1, 9, O, Ip * wide, device=DEV, dtype=H16)
    b = torch.zeros(O, device=DEV)
    y = torch.zeros(N, H, W, O * wide, device=DEV, dtype=H16)
    L, P = capi.lib(), capi.ptr
    if split:
        return lambda: L.r3dp_sr_tcx_conv(P(x, H16), P(wp, H16), P(b), N, 1, I, O, H, W, ksize, act, P(y, H16), capi.stream())
    return lambda: L.r3dp_sr_tc_conv_res(P(x, H16), P(wp, H16), P(b), N, 1, I, O, H, W, ksize, act, None, P(y, H16), capi.stream())


def _gate_call(stride, lo_off):
    N, H, W = 1, 4, 8
    y = torch.zeros(N * H * W * stride + stride, device=DEV, dtype=H16)
    cap, out = torch.ones(N, 1, H, W, device=DEV), torch.zeros(N, 1, H, W, device=DEV)
    return lambda: capi.lib().r3dp_sr_alpha_gate(capi.ptr(y, H16), stride, lo_off, capi.ptr(cap), N, H, W, capi.ptr(out), capi.stream())


REJECTED = {
    'layer_W96': (lambda s: _layer_call(s, W=96), 'W % 128 == 0'),
    'layer_up2_W96': (lambda s: _layer_call(s, W=96, up=2), 'W % 128 == 0'),
    'layer_Cout192': (lambda s: _layer_call(s, O=192), 'Cout % 128 == 0'),
    'layer_Cout384': (lambda s: _layer_call(s, O=384), 'Cout == 128 or Cout == 256'),
    'layer_up2_Cout384': (lambda s: _layer_call(s, O=384, up=2), 'Cout == 128 or Cout == 256'),
    'layer_Nw3_of_2': (lambda s: _layer_call(s, Nw=3), 'Nw == N or Nw == 1'),
    'layer_up3': (lambda s: _layer_call(s, up=3), 'up must be 1 or 2'),
    'layer_up2_I320': (lambda s: _layer_call(s, I=320, up=2), 'at most 256 input channels'),
    'layer_torgb_H5': (lambda s: _fused_call('layer_torgb', s, H=5), 'H % 2 == 0'),
    'layer_torgb_Cout384': (lambda s: _fused_call('layer_torgb', s, O=384), 'Cout 128 or 256'),
    'last_layer_H5': (lambda s: _fused_call('last_layer', s, O=128, H=5), 'H % 2 == 0'),
    'last_layer_Nw3_of_2': (lambda s: _fused_call('last_layer', s, Nw=3), 'Nw == N or Nw == 1'),
    'conv_ksize2': (lambda s: _conv_call(s, ksize=2), 'ksize must be 1 or 3'),
    'conv_act4': (lambda s: _conv_call(s, act=4), 'act must be 0..3'),
    'conv_W96': (lambda s: _conv_call(s, W=96), 'W % 128 == 0'),
}


@pytest.mark.parametrize('split', [False, True], ids=['tc', 'tcx'])
@pytest.mark.parametrize('case', list(REJECTED))
def test_rejected_calls_launch_nothing(case, split):
    make, needle = REJECTED[case]
    _expect_rejected(make(split), needle)


def test_alpha_gate_rejects_lo_off_at_stride():
    _expect_rejected(_gate_call(8, 8), '0 <= lo_off < stride')
    _expect_rejected(_gate_call(8, 9), '0 <= lo_off < stride')


if __name__ == '__main__':
    torch.save(_variant_outputs(), sys.argv[1])
