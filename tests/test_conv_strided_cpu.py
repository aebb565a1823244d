"""Host-only checks of the strided convolution backward passes: the strided backward oracles (tests/conv_strided_oracle.py)
against the stride-1 oracles of oracle/lenet_oracle.c and against its strided forward oracle through the adjoint identities, and
the tile planning of pcnn_conv_bwd_plan_info_strided (pure host logic)."""
import ctypes as C

import numpy as np
import pytest

import conv_strided_oracle as SO
import oracle_lib as O


def _oracle_case(rng, N, H, W, Cin, K, R, S, stride):
    P, Q = (H - R) // stride + 1, (W - S) // stride + 1
    x = rng.uniform(0, 1, (N, H, W, Cin)).astype(np.float32)
    dy = rng.uniform(-1, 1, (N, P, Q, K)).astype(np.float32)
    f = rng.uniform(-0.5, 0.5, (K, R, S, Cin)).astype(np.float32)
    return x, dy, f, P, Q


@pytest.mark.parametrize("shape", [(2, 9, 11, 3, 5, 3, 3), (1, 12, 10, 1, 4, 5, 5), (3, 7, 8, 2, 3, 3, 2)])
def test_strided_oracles_at_stride_1_are_the_stride_1_oracles(shape):
    N, H, W, Cin, K, R, S = shape
    x, dy, f, _, _ = _oracle_case(np.random.default_rng(sum(shape)), N, H, W, Cin, K, R, S, 1)
    L = O.oracle()
    dw1 = np.empty((K, R, S, Cin), np.float32)
    L.orc_conv_wgrad_nhwc(O.fp(x.reshape(-1)), O.fp(dy.reshape(-1)), O.fp(dw1.reshape(-1)), N, H, W, Cin, K, R, S)
    dws = SO.conv_wgrad_nhwc_strided(x, dy, R, S, 1)
    assert np.array_equal(dw1.view(np.uint32), dws.view(np.uint32))
    dx1 = np.empty((N, H, W, Cin), np.float32)
    L.orc_conv_dgrad_nhwc(O.fp(dy.reshape(-1)), O.fp(f.reshape(-1)), O.fp(dx1.reshape(-1)), N, H, W, Cin, K, R, S)
    dxs = SO.conv_dgrad_nhwc_strided(dy, f, H, W, 1)
    assert np.array_equal(dx1.view(np.uint32), dxs.view(np.uint32))


@pytest.mark.parametrize("shape", [(2, 11, 13, 3, 4, 3, 3, 2),     # (H - R) and (W - S) odd: the last row / column no tap reaches
                                   (1, 14, 12, 1, 5, 5, 5, 2),
                                   (2, 13, 16, 2, 3, 3, 3, 3),     # 10 % 3, 13 % 3 != 0
                                   (1, 17, 15, 3, 4, 3, 3, 4),     # S < stride: columns between windows
                                   (1, 12, 19, 2, 6, 5, 3, 4),
                                   (1, 16, 16, 1, 3, 7, 7, 3)])
def test_strided_backward_oracles_are_adjoint_to_the_strided_forward_oracle(shape):
    """<fwd(x, f), dy> = <f, wgrad(x, dy)> = <x, dgrad(dy, f)> with bias 0: pins both new oracles to orc_conv_fwd_nhwc_strided."""
    N, H, W, Cin, K, R, S, stride = shape
    x, dy, f, P, Q = _oracle_case(np.random.default_rng(sum(shape)), N, H, W, Cin, K, R, S, stride)
    L = O.oracle()
    y = np.empty((N, P, Q, K), np.float32)
    L.orc_conv_fwd_nhwc_strided(O.fp(x.reshape(-1)), O.fp(f.reshape(-1)), O.fp(np.zeros(K, np.float32)), O.fp(y.reshape(-1)),
                                N, H, W, Cin, K, R, S, stride)
    dw = SO.conv_wgrad_nhwc_strided(x, dy, R, S, stride)
    dx = SO.conv_dgrad_nhwc_strided(dy, f, H, W, stride)
    a = float(np.dot(y.astype(np.float64).ravel(), dy.astype(np.float64).ravel()))
    b = float(np.dot(f.astype(np.float64).ravel(), dw.astype(np.float64).ravel()))
    c = float(np.dot(x.astype(np.float64).ravel(), dx.astype(np.float64).ravel()))
    scale = np.abs(y.astype(np.float64) * dy).sum()
    assert abs(a - b) <= 1e-6 * scale and abs(a - c) <= 1e-6 * scale, (a, b, c, scale)
    # rows and columns no window reaches get zero gradient
    hmax, wmax = (P - 1) * stride + R, (Q - 1) * stride + S
    assert np.all(dx[:, hmax:] == 0) and np.all(dx[:, :, wmax:] == 0)
    if S < stride:
        cols = np.arange(W)
        assert np.all(dx[:, :, (cols % stride) >= S] == 0)


def _info(pkg, *shape, strided=True):
    out = (C.c_int * 9)()
    fn = pkg.lib().pcnn_conv_bwd_plan_info_strided if strided else pkg.lib().pcnn_conv_bwd_plan_info
    assert fn(*shape, out) == 0
    return list(out)


def test_strided_backward_tile_planning_is_host_logic(pkg):
    # stride 1 is the existing query, for the shapes its own test pins
    for shape in [(128, 224, 224, 3, 64, 3, 3), (4, 64, 64, 3, 128, 3, 3), (4, 28, 28, 1, 6, 5, 5), (1, 32, 32, 3, 320, 3, 3),
                  (1, 32, 32, 3, 64, 5, 5)]:
        assert _info(pkg, *shape, 1) == _info(pkg, *shape, strided=False), shape
    # config 5 at stride 2 (P = Q = 111): both passes on the tensor cores; 3 dy rows = 7 x rows = 63 Hankel rows, one chunk of 112 pixels
    cfg5 = _info(pkg, 128, 224, 224, 3, 64, 3, 3, 2)
    assert cfg5[:3] == [1, 3, 112] and cfg5[3] >= 2
    assert cfg5[4] == 1 and cfg5[5] == 1 and cfg5[6] == 56       # one strip of 224 columns: 28 dy pixels = 56 dx columns per quarter
    # 5x5x3 at stride 2: 5 x rows x 15 = 75 Hankel rows > 64 even for one dy row per tile; the input gradient is built
    s553 = _info(pkg, 1, 20, 40, 3, 64, 5, 5, 2)
    assert s553[0] == 0 and s553[4] == 1
    # 3x3x8 at stride 3: no input-gradient kernel instantiated
    assert _info(pkg, 1, 24, 24, 8, 64, 3, 3, 3)[4] == 0
    # the minimum set of input-gradient kernels is built
    for (R, S, Cin, st) in [(3, 3, c, 2) for c in (1, 2, 3, 4, 8)] + [(5, 5, 1, 2), (5, 5, 3, 2), (7, 7, 1, 2)] + \
                           [(3, 3, c, 3) for c in (1, 2, 3)] + [(3, 3, 3, 4), (5, 5, 1, 4)]:
        assert _info(pkg, 1, 40, 48, Cin, 64, R, S, st)[4] == 1, (R, S, Cin, st)
    # window steps outside 1..4 are argument errors
    out = (C.c_int * 9)()
    for bad in (0, 5, -1):
        assert pkg.lib().pcnn_conv_bwd_plan_info_strided(1, 32, 32, 3, 64, 3, 3, bad, out) != 0
