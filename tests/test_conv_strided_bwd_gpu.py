"""GPU parity tests of the strided convolution backward passes (pcnn_conv_wgrad_strided / pcnn_conv_dgrad_strided): the tcgen05
kernels of csrc/conv_wgrad_tc.cu and csrc/conv_dgrad_tc.cu and the FMA-pipe kernels of csrc/conv_bwd.cu, against
the strided backward oracles of tests/conv_strided_oracle.py on the same bf16-rounded operands.  Bounds as for stride 1:
    wgrad (fp32 out) rel-L2 <= 1e-5;  dgrad (bf16 out) |d| <= 2^-8 |ref| + 1e-3 per element.
"""
import ctypes as C

import numpy as np
import pytest

import conv_strided_oracle as SO
import oracle_lib as O

pytestmark = pytest.mark.gpu

CANARY = 0x7FC0                     # bf16 NaN: every dx element must be overwritten


def operands(pkg, rng, N, H, W, Cin, K, R, S, stride):
    P, Q = (H - R) // stride + 1, (W - S) // stride + 1
    x = pkg.bf16_bits_to_f32(pkg.f32_to_bf16_bits(rng.uniform(0, 1, (N, H, W, Cin)).astype(np.float32)))
    dy = pkg.bf16_bits_to_f32(pkg.f32_to_bf16_bits(rng.uniform(-1, 1, (N, P, Q, K)).astype(np.float32)))
    f = pkg.bf16_bits_to_f32(pkg.f32_to_bf16_bits(rng.uniform(-0.5, 0.5, (K, R, S, Cin)).astype(np.float32)))
    return x, dy, f


def oracles(x, dy, f, stride):
    _, H, W, _ = x.shape
    _, R, S, _ = f.shape
    return SO.conv_wgrad_nhwc_strided(x, dy, R, S, stride), SO.conv_dgrad_nhwc_strided(dy, f, H, W, stride)


def pitched(pkg, a, pitch):
    """NHWC float32 -> bf16 rows [N][H][pitch] (pad elements 0)"""
    N, H, W, Cin = a.shape
    out = np.zeros((N, H, pitch), np.uint16)
    out[:, :, : W * Cin] = pkg.f32_to_bf16_bits(a).reshape(N, H, W * Cin)
    return out


def rel_l2(got, ref):
    return np.linalg.norm((got - ref).astype(np.float64)) / np.linalg.norm(ref.astype(np.float64))


def dgrad_ok(got, ref):
    return np.all(np.abs(got - ref) <= 2.0 ** -8 * np.abs(ref) + 1e-3)


def plan_info(pkg, N, H, W, Cin, K, R, S, stride):
    out = (C.c_int * 9)()
    assert pkg.lib().pcnn_conv_bwd_plan_info_strided(N, H, W, Cin, K, R, S, stride, out) == 0
    return list(out)


STRIDED_SHAPES = [(3, 28, 28, 1, 16, 5, 5, 2),       # the strided forward test shapes ...
                  (2, 64, 40, 3, 64, 3, 3, 2),
                  (1, 224, 224, 3, 64, 3, 3, 2),     # config 5 at stride 2
                  (2, 33, 30, 2, 32, 3, 3, 3),       # stride 3, 33 rows per image (not a multiple of 3)
                  (1, 30, 32, 1, 64, 5, 5, 2),       # last row and column reached by no tap
                  (1, 40, 48, 1, 64, 7, 7, 2),       # 7x7 taps
                  (2, 24, 32, 3, 128, 3, 3, 2),      # two filter groups
                  (4, 28, 28, 1, 6, 5, 5, 2),        # 6 filters: padded dy copy
                  (1, 26, 30, 3, 64, 3, 3, 4),       # S < stride: columns between the windows are zero
                  (1, 20, 40, 3, 64, 5, 5, 2)]       # weight gradient refused (75 Hankel rows), input gradient on the tensor cores


@pytest.mark.parametrize("shape", STRIDED_SHAPES)
def test_strided_wgrad_and_dgrad_vs_oracle_and_fma_path(eng, pkg, shape):
    N, H, W, Cin, K, R, S, stride = shape
    rng = np.random.default_rng(sum(shape) + 7)
    x, dy, f = operands(pkg, rng, N, H, W, Cin, K, R, S, stride)
    dw_ref, dx_ref = oracles(x, dy, f, stride)
    pitch = (W * Cin + 7) // 8 * 8                    # the tensor-core weight gradient needs a pitch that is a multiple of 8
    info = plan_info(pkg, N, H, W, Cin, K, R, S, stride)
    wgrad_tc, dgrad_tc = bool(info[0]), bool(info[4])
    assert dgrad_tc
    xd, dyd, fd = eng.to_device(pitched(pkg, x, pitch)), eng.to_device(pkg.f32_to_bf16_bits(dy)), eng.to_device(f)
    res = {}
    try:
        for path in ("tc", "fma"):
            eng.conv_bwd_select(reference=(path == "fma"))
            l0 = eng.launch_count()
            dw = eng.array((K, R, S, Cin))
            got_w = None
            if path == "fma" or wgrad_tc:
                eng.conv_wgrad(xd, dyd, dw, N, H, W, Cin, K, R, S, row_pitch=pitch, stride=stride)
                got_w = dw.to_host()
                assert rel_l2(got_w, dw_ref) <= 1e-5, path
                eng.conv_wgrad(xd, dyd, dw, N, H, W, Cin, K, R, S, row_pitch=pitch, stride=stride)
                assert np.array_equal(dw.to_host().view(np.uint32), got_w.view(np.uint32)), path       # deterministic
            else:                                     # no tensor-core weight gradient for this shape: refused, not rerouted
                with pytest.raises(pkg.PcnnError, match="pcnn_conv_bwd_select"):
                    eng.conv_wgrad(xd, dyd, dw, N, H, W, Cin, K, R, S, row_pitch=pitch, stride=stride)
            dxo = eng.to_device(np.full((N, H, pitch), CANARY, np.uint16))
            eng.conv_dgrad(dyd, fd, dxo, N, H, W, Cin, K, R, S, row_pitch=pitch, stride=stride)
            raw = dxo.to_host()
            got_x = pkg.bf16_bits_to_f32(raw[:, :, : W * Cin].reshape(N, H, W, Cin))
            assert np.isfinite(got_x).all(), path
            assert dgrad_ok(got_x, dx_ref), (path, float(np.abs(got_x - dx_ref).max()))
            eng.conv_dgrad(dyd, fd, dxo, N, H, W, Cin, K, R, S, row_pitch=pitch, stride=stride)
            assert np.array_equal(dxo.to_host(), raw), path                                               # deterministic
            res[path] = (got_w, eng.launch_count() - l0)
    finally:
        eng.conv_bwd_select(reference=False)
    assert res["tc"][1] != res["fma"][1]              # different kernels ran
    if wgrad_tc:
        assert rel_l2(res["tc"][0], res["fma"][0]) <= 1e-5


def test_strided_shape_without_tensor_core_kernel_is_refused_and_fma_path_computes_it(eng, pkg):
    N, H, W, Cin, K, R, S, stride = 1, 24, 24, 8, 64, 3, 3, 3        # 3x3x8 at stride 3: neither pass has a tensor-core kernel
    rng = np.random.default_rng(3)
    x, dy, f = operands(pkg, rng, N, H, W, Cin, K, R, S, stride)
    dw_ref, dx_ref = oracles(x, dy, f, stride)
    xd, dyd, fd = eng.to_device(pkg.f32_to_bf16_bits(x)), eng.to_device(pkg.f32_to_bf16_bits(dy)), eng.to_device(f)
    dw, dxo = eng.array((K, R, S, Cin)), eng.array((N, H, W, Cin), np.uint16)
    with pytest.raises(pkg.PcnnError, match="pcnn_conv_bwd_select"):
        eng.conv_wgrad(xd, dyd, dw, N, H, W, Cin, K, R, S, stride=stride)
    with pytest.raises(pkg.PcnnError, match="pcnn_conv_bwd_select"):
        eng.conv_dgrad(dyd, fd, dxo, N, H, W, Cin, K, R, S, stride=stride)
    with pytest.raises(pkg.PcnnError):
        eng.conv_dgrad(dyd, fd, dxo, N, H, W, Cin, K, R, S, stride=5)
    eng.conv_bwd_select(reference=True)
    try:
        eng.conv_wgrad(xd, dyd, dw, N, H, W, Cin, K, R, S, stride=stride)
        eng.conv_dgrad(dyd, fd, dxo, N, H, W, Cin, K, R, S, stride=stride)
    finally:
        eng.conv_bwd_select(reference=False)
    assert rel_l2(dw.to_host(), dw_ref) <= 1e-5
    assert dgrad_ok(pkg.bf16_bits_to_f32(dxo.to_host()), dx_ref)


def test_stride_1_through_the_strided_entry_points_is_bit_identical(eng, pkg):
    N, H, W, Cin, K, R, S = 2, 40, 40, 3, 64, 3, 3
    rng = np.random.default_rng(17)
    x, dy, f = operands(pkg, rng, N, H, W, Cin, K, R, S, 1)
    xd, dyd, fd = eng.to_device(pkg.f32_to_bf16_bits(x)), eng.to_device(pkg.f32_to_bf16_bits(dy)), eng.to_device(f)
    try:
        for path in ("tc", "fma"):
            eng.conv_bwd_select(reference=(path == "fma"))
            dw1, dws = eng.array((K, R, S, Cin)), eng.array((K, R, S, Cin))
            dx1, dxs = eng.array((N, H, W, Cin), np.uint16), eng.array((N, H, W, Cin), np.uint16)
            eng.conv_wgrad(xd, dyd, dw1, N, H, W, Cin, K, R, S)
            eng._call("pcnn_conv_wgrad_strided", xd.ptr, dyd.ptr, dws.ptr, N, H, W, Cin, K, R, S, 1, 0, 0)
            eng.conv_dgrad(dyd, fd, dx1, N, H, W, Cin, K, R, S)
            eng._call("pcnn_conv_dgrad_strided", dyd.ptr, fd.ptr, dxs.ptr, N, H, W, Cin, K, R, S, 1, 0, 0)
            assert np.array_equal(dw1.to_host().view(np.uint32), dws.to_host().view(np.uint32)), path
            assert np.array_equal(dx1.to_host(), dxs.to_host()), path
    finally:
        eng.conv_bwd_select(reference=False)


def test_strided_dgrad_honours_row_and_image_pitch(eng, pkg):
    """dx at stride 2 written into a padded canvas (row pitch 128 elements, 48 rows per image): pad elements keep their contents."""
    N, H, W, Cin, K, R, S, stride = 2, 40, 40, 3, 64, 3, 3, 2
    rng = np.random.default_rng(5)
    _, dy, f = operands(pkg, rng, N, H, W, Cin, K, R, S, stride)
    dx_ref = SO.conv_dgrad_nhwc_strided(dy, f, H, W, stride)
    pitch, rows = 128, 48
    dxo = eng.to_device(np.full((N, rows, pitch), 0x4242, np.uint16))
    eng.conv_dgrad(eng.to_device(pkg.f32_to_bf16_bits(dy)), eng.to_device(f), dxo, N, H, W, Cin, K, R, S, row_pitch=pitch, image_rows=rows,
                   stride=stride)
    out = dxo.to_host().reshape(N, rows, pitch)
    got = pkg.bf16_bits_to_f32(out[:, :H, :W * Cin].reshape(N, H, W, Cin))
    assert dgrad_ok(got, dx_ref)
    assert np.all(out[:, H:, :] == 0x4242) and np.all(out[:, :, W * Cin:] == 0x4242)


def test_same_padded_stride_2_layer_through_pad_and_crop(eng, pkg):
    """A 'same'-padded 3x3/2 layer (32x32x3 -> 16x16x64): pad -> strided forward plan -> strided weight and input gradient -> crop,
    against the strided oracles on the host-padded tensors."""
    N, H, W, Cin, K, R, S, pad, stride = 2, 32, 32, 3, 64, 3, 3, 1, 2
    Hp, Wp = H + 2 * pad, W + 2 * pad                         # 34 rows per image: a multiple of the stride, as the forward plan needs
    P, Q = (Hp - R) // stride + 1, (Wp - S) // stride + 1
    assert (P, Q) == (16, 16)
    rng = np.random.default_rng(23)
    x = pkg.bf16_bits_to_f32(pkg.f32_to_bf16_bits(rng.uniform(0, 1, (N, H, W, Cin)).astype(np.float32)))
    f = pkg.bf16_bits_to_f32(pkg.f32_to_bf16_bits(rng.uniform(-0.5, 0.5, (K, R, S, Cin)).astype(np.float32)))
    dy = pkg.bf16_bits_to_f32(pkg.f32_to_bf16_bits(rng.uniform(-1, 1, (N, P, Q, K)).astype(np.float32)))
    xp = np.zeros((N, Hp, Wp, Cin), np.float32)
    xp[:, pad:pad + H, pad:pad + W, :] = x
    y_ref = np.empty((N, P, Q, K), np.float32)
    O.oracle().orc_conv_fwd_nhwc_strided(O.fp(xp.reshape(-1)), O.fp(f.reshape(-1)), O.fp(np.zeros(K, np.float32)), O.fp(y_ref.reshape(-1)),
                                         N, Hp, Wp, Cin, K, R, S, stride)
    dw_ref, dxp_ref = oracles(xp, dy, f, stride)
    pitch = (Wp * Cin + 7) // 8 * 8
    canvas = eng.to_device(np.full((N, Hp, pitch), 0x4242, np.uint16))
    eng.pad_nhwc(eng.to_device(pkg.f32_to_bf16_bits(x)), canvas, N, H, W, Cin, pad, pad, dst_row_pitch=pitch)
    plan = pkg.ConvPlan(eng, N, Hp, Wp, Cin, K, R, S, f, None, act=0, row_pitch=pitch, stride=stride)
    yd = eng.array((N, P, Q, K), np.uint16)
    plan.fwd(canvas, yd)
    got_y = pkg.bf16_bits_to_f32(yd.to_host())
    plan.close()
    assert dgrad_ok(got_y, y_ref)
    dyd = eng.to_device(pkg.f32_to_bf16_bits(dy))
    dw = eng.array((K, R, S, Cin))
    eng.conv_wgrad(canvas, dyd, dw, N, Hp, Wp, Cin, K, R, S, row_pitch=pitch, stride=stride)
    assert rel_l2(dw.to_host(), dw_ref) <= 1e-5
    dxp = eng.to_device(np.full((N, Hp, pitch), CANARY, np.uint16))
    eng.conv_dgrad(dyd, eng.to_device(f), dxp, N, Hp, Wp, Cin, K, R, S, row_pitch=pitch, stride=stride)
    dxc = eng.array((N, H, W, Cin), np.uint16)
    eng.crop_nhwc(dxp, dxc, N, H, W, Cin, pad, pad, src_row_pitch=pitch)
    got_dx = pkg.bf16_bits_to_f32(dxc.to_host())
    assert np.isfinite(got_dx).all()
    assert dgrad_ok(got_dx, dxp_ref[:, pad:pad + H, pad:pad + W, :])
