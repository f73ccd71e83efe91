"""The split-operand SR convolutions (`sr_mode='tc_exact'`, csrc/sr_tc.cu conv_tc3_kernel<R, true>) claim fp32-grade results from fp16 tensor-core
operands: weights are stored x 2^10 and split as w = hi + lo, activations are split WITHOUT scaling, the K loop accumulates hi*hi + lo*hi + hi*lo
in fp32 and the epilogue multiplies by 2^-10.  This CPU test restates that arithmetic with numpy on one 256-channel 3x3 layer (K = 2304) and
bounds its error against float64, next to an fp32 evaluation of the same product.  Unscaled activations have a range floor: once |x| falls
below about 2^-4 the lo halves become fp16 subnormals and the error grows.  The GPU kernel tests (test_gpu_sr_kernels.py) hold the split
path to fp32 grade, so the scale of their activations must stay inside that band."""
import numpy as np
import pytest

WEIGHT_SCALE = 2.0 ** 10          # kSplitWeightScale
K = 2304                          # 256 channels x 9 taps
FP32_GRADE_MIN_SCALE = 2.0 ** -4  # smallest input scale at which the split product is within 2x of fp32


def _split(v):
    hi = v.astype(np.float16)
    lo = (v - hi.astype(np.float32)).astype(np.float16)
    return hi.astype(np.float32), lo.astype(np.float32)


def _conv_split(x, w):
    """x [M,K] fp32 (im2col rows), w [O,K] fp32 -> the kernel's product: three fp16 partial products summed in fp32, then x 2^-10."""
    xh, xl = _split(x)
    wh, wl = _split((w * np.float32(WEIGHT_SCALE)).astype(np.float32))
    acc = (xh @ wh.T).astype(np.float32) + (xl @ wh.T).astype(np.float32) + (xh @ wl.T).astype(np.float32)
    return (acc * np.float32(1.0 / WEIGHT_SCALE)).astype(np.float32)


def _errors(scale, seed=0, M=512, O=128):
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((M, K)) * scale).astype(np.float32)
    w = (rng.standard_normal((O, K)) / np.sqrt(K)).astype(np.float32)            # demodulated weights: unit-norm filters
    y64 = x.astype(np.float64) @ w.astype(np.float64).T
    ymax = float(np.abs(y64).max())
    e_split = float(np.abs(_conv_split(x, w) - y64).max()) / ymax
    e_f32 = float(np.abs((x @ w.T).astype(np.float32) - y64).max()) / ymax
    e_f16 = float(np.abs(x.astype(np.float16).astype(np.float32) @ w.astype(np.float16).astype(np.float32).T - y64).max()) / ymax
    return e_split, e_f32, e_f16


def _rel_split_error(v):
    hi, lo = _split(v)
    return np.abs((hi.astype(np.float64) + lo) - v) / np.abs(v)


def test_weight_scale_keeps_the_split_at_22_bits():
    """Why the weights carry 2^10: demodulated 3x3 weights of a 256-channel layer are O(1/48); unscaled, their lo halves (~2^-17) fall into
    the fp16 subnormals (resolution 2^-24) and hi + lo loses bits.  Scaled, every weight above 2^-10 is reconstructed to 2^-21."""
    rng = np.random.default_rng(3)
    w = (rng.standard_normal(1 << 16) / np.sqrt(K)).astype(np.float32)
    w = w[np.abs(w) > 2.0 ** -10]
    assert _rel_split_error((w * np.float32(WEIGHT_SCALE)).astype(np.float32)).max() <= 2.0 ** -21
    assert _rel_split_error(w).max() > 2.0 ** -16


@pytest.mark.parametrize('log2_scale', [0, -2, -4])
def test_split_conv_is_fp32_grade_in_its_range(log2_scale):
    e_split, e_f32, e_f16 = _errors(2.0 ** log2_scale)
    print(f'input scale 2^{log2_scale}: split {e_split:.2e}, fp32 {e_f32:.2e}, fp16 operands {e_f16:.2e} (max error / max|y|)')
    assert e_split <= 2.0 * e_f32
    assert e_f16 > 50.0 * e_split


def test_split_conv_degrades_below_its_range():
    """Documents the floor rather than hiding it: at 2^-10 the unscaled activations' lo halves are subnormal and the split product is no
    longer within 2x of fp32 (still well ahead of plain fp16 operands)."""
    e_split, e_f32, e_f16 = _errors(2.0 ** -10)
    print(f'input scale 2^-10: split {e_split:.2e}, fp32 {e_f32:.2e}, fp16 operands {e_f16:.2e}')
    assert e_split > 2.0 * e_f32
    assert e_split < 1e-4 < e_f16


def test_gpu_test_inputs_lie_in_the_fp32_grade_band():
    from test_gpu_sr_kernels import ACT_SCALE
    assert ACT_SCALE >= FP32_GRADE_MIN_SCALE
    e_split, e_f32, _ = _errors(ACT_SCALE)
    assert e_split <= 2.0 * e_f32
