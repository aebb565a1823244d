"""Direct restatements of the two backward passes of orc_conv_fwd_nhwc_strided (oracle/lenet_oracle.c), window step `stride`,
P = (H-R)/stride + 1, Q = (W-S)/stride + 1, NHWC activations, KRSC filters:

    dw[k][r][s][c] = sum_{n,p,q} dy[n][p][q][k] * x[n][p*stride+r][q*stride+s][c]
    dx[n][h][w][c] = sum over (h-r) % stride == 0, (w-s) % stride == 0 of dy[n][(h-r)/stride][(w-s)/stride][k] * f[k][r][s][c]

Double accumulation, one float32 rounding at the end.  Every output element receives its terms in the order of the C oracles
orc_conv_wgrad_nhwc / orc_conv_dgrad_nhwc ((n, p, q) for the weight gradient, (r, s, k) for the input gradient; the products of
two float32 values are exact in double), so at stride 1 the results are bit-identical to theirs.  The loops run over the
reduction indices and the arithmetic is vectorised over the outputs."""
import numpy as np


def conv_wgrad_nhwc_strided(x, dy, R, S, stride):
    """x [N][H][W][C], dy [N][P][Q][K] (float32) -> dw [K][R][S][C] float32"""
    x = np.asarray(x, np.float64)
    dy = np.asarray(dy, np.float64)
    N, P, Q, K = dy.shape
    acc = np.zeros((K, R, S, x.shape[3]))
    for n in range(N):
        for p in range(P):
            for q in range(Q):
                win = x[n, p * stride:p * stride + R, q * stride:q * stride + S, :]
                acc += dy[n, p, q, :, None, None, None] * win[None]
    return acc.astype(np.float32)


def conv_dgrad_nhwc_strided(dy, f, H, W, stride):
    """dy [N][P][Q][K], f [K][R][S][C] (float32) -> dx [N][H][W][C] float32 (0 where no tap reaches)"""
    dy = np.asarray(dy, np.float64)
    f = np.asarray(f, np.float64)
    N, P, Q, K = dy.shape
    _, R, S, C = f.shape
    acc = np.zeros((N, H, W, C))
    for r in range(R):
        for s in range(S):
            rows = slice(r, r + (P - 1) * stride + 1, stride)
            cols = slice(s, s + (Q - 1) * stride + 1, stride)
            for k in range(K):
                acc[:, rows, cols, :] += dy[:, :, :, k, None] * f[k, r, s][None, None, None, :]
    return acc.astype(np.float32)
