"""ctypes access to the parity checkers under oracle/ (TEST INFRASTRUCTURE ONLY).

`oracle()` loads oracle/liblenet_oracle.so, the C restatement of /root/reference/Sequential/layer.h + Main.cpp.
`reference()` loads oracle/_ref/libref_seq.so, the unmodified reference compiled where it lies (None when absent).
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this module.
"""
import ctypes as C
import hashlib
import os
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_SO = os.path.join(ROOT, "oracle", "liblenet_oracle.so")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libref_seq.so")
REF_NATIVE_SO = os.path.join(ROOT, "oracle", "_ref", "libref_seq_native.so")   # -O3 -march=x86-64-v3: timing only
REF_DATA = os.path.join(ROOT, "oracle", "_ref", "data")
GOLDEN = os.path.join(ROOT, "tests", "golden")

NPARAM = 2343
N_ACTS = 3456 * 2 + 216 * 2 + 10 * 2          # 7364
OFF = dict(c1w=(0, 150), c1b=(150, 156), s1w=(156, 172), s1b=(172, 173), fw=(173, 2333), fb=(2333, 2343))
ACT_OFF = dict(c1_pre=(0, 3456), c1_out=(3456, 6912), s1_pre=(6912, 7128), s1_out=(7128, 7344),
               f_pre=(7344, 7354), f_out=(7354, 7364))
# orc_back struct layout (floats)
N_BACK = 7355 + NPARAM
BACK_OFF = dict(f_dpre=(0, 10), s1_dout=(10, 226), s1_dpre=(226, 442), c1_dout=(442, 3898),
                c1_dpre=(3898, 7354), g=(7354, 7354 + NPARAM), err=(7354 + NPARAM, 7355 + NPARAM))

_f = C.POINTER(C.c_float)
_d = C.POINTER(C.c_double)
_u8 = C.POINTER(C.c_uint8)
_i32 = C.POINTER(C.c_int32)


def fp(a):
    assert a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_f)


def dp(a):
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_d)


def u8p(a):
    assert a.dtype == np.uint8 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_u8)


def i32p(a):
    assert a.dtype == np.int32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_i32)


_oracle = None
_ref = None
_ref_native = None


def oracle():
    global _oracle
    if _oracle is None:
        if not os.path.exists(ORACLE_SO):
            raise RuntimeError(f"{ORACLE_SO} missing: run `make -C oracle` (or __graft_entry__.build())")
        L = C.CDLL(ORACLE_SO)
        L.orc_sigmoid.restype = C.c_float
        L.orc_sigmoid.argtypes = [C.c_float]
        L.orc_vector_norm.restype = C.c_float
        L.orc_bias_sum_s1.restype = C.c_float
        L.orc_train_step.restype = C.c_float
        L.orc_train_step.argtypes = [_f, _f, C.c_uint]
        L.orc_learn.restype = C.c_float
        L.orc_learn.argtypes = [_f, _u8, _u8, C.c_long]
        L.orc_test.restype = C.c_long
        L.orc_test.argtypes = [_f, _u8, _u8, C.c_long]
        L.orc_classify.restype = C.c_uint
        L.orc_u8_to_f32.argtypes = [_u8, _f, C.c_long]
        L.orc_batch_grad.argtypes = [_f, _f, _u8, C.c_long, _d, _d]
        L.orc_apply_update.argtypes = [_f, _f, C.c_float]
        L.orc_backward.argtypes = [_f, _f, C.c_uint, C.c_void_p, C.c_void_p]
        L.orc_forward.argtypes = [_f, _f, C.c_void_p]
        L.orc_softmax_ce.restype = C.c_float
        L.orc_softmax_ce.argtypes = [_f, C.c_uint, C.c_int, _f, _f]
        L.orc_maxpool_fwd.argtypes = [_f, _f, _i32, C.c_int, C.c_int, C.c_int, C.c_int]
        L.orc_maxpool_bwd.argtypes = [_f, _i32, _f, C.c_int, C.c_int, C.c_int, C.c_int]
        L.orc_conv_fwd_nhwc.argtypes = [_f, _f, _f, _f] + [C.c_int] * 7
        L.orc_conv_fwd_nhwc_strided.argtypes = [_f, _f, _f, _f] + [C.c_int] * 8
        L.orc_conv_wgrad_nhwc.argtypes = [_f, _f, _f] + [C.c_int] * 7
        L.orc_conv_dgrad_nhwc.argtypes = [_f, _f, _f] + [C.c_int] * 7
        assert L.orc_sizeof_acts() == N_ACTS * 4
        assert L.orc_sizeof_back() == N_BACK * 4
        _oracle = L
    return _oracle


def reference(native=False):
    """The unmodified reference, or None when oracle/_ref was not built (no /root/reference at build time).
    native=True: the same sources built -O3 with FMA contraction (bench.py's best-CPU timing; NOT a parity checker)."""
    global _ref, _ref_native
    if native:
        if _ref_native is None and os.path.exists(REF_NATIVE_SO):
            L = C.CDLL(REF_NATIVE_SO)
            L.ref_learn_loop_u8.restype = C.c_float
            L.ref_learn_loop_u8.argtypes = [_u8, _u8, C.c_long, _d]
            _ref_native = L
        return _ref_native
    if _ref is None:
        if not os.path.exists(REF_SO):
            return None
        L = C.CDLL(REF_SO)
        L.ref_train_step_u8.restype = C.c_float
        L.ref_train_step_u8.argtypes = [_u8, C.c_uint]
        L.ref_learn_loop_u8.restype = C.c_float
        L.ref_learn_loop_u8.argtypes = [_u8, _u8, C.c_long, _d]
        L.ref_learn_driver_u8.argtypes = [_u8, _u8, C.c_long]
        L.ref_test_u8.restype = C.c_long
        L.ref_test_u8.argtypes = [_u8, _u8, C.c_long]
        L.ref_classify_u8.restype = C.c_uint
        L.ref_step_function.restype = C.c_float
        L.ref_step_function.argtypes = [C.c_float]
        L.ref_vectorNorm.restype = C.c_float
        _ref = L
    return _ref


# ---------------------------------------------------------------- LeNet-5-style variant (oracle/lenet5_oracle.c; parity unpinned)
L5_SO = os.path.join(ROOT, "oracle", "liblenet5_oracle.so")
L5_NPARAM = 5152
L5_OFF = dict(c1w=(0, 150), c1b=(150, 156), s2w=(156, 160), s2b=(160, 161), c3w=(161, 2561), c3b=(2561, 2577), s4w=(2577, 2581),
              s4b=(2581, 2582), fw=(2582, 5142), fb=(5142, 5152))
_l5 = None


def lenet5():
    global _l5
    if _l5 is None:
        if not os.path.exists(L5_SO):
            raise RuntimeError(f"{L5_SO} missing: run `make -C oracle` (or __graft_entry__.build())")
        L = C.CDLL(L5_SO)
        assert L.l5_nparam() == L5_NPARAM
        L.l5_init_params.argtypes = [_f, C.c_uint32]
        L.l5_batch_grad.argtypes = [_f, _f, _u8, C.c_long, _d, _d]
        L.l5_apply_update.argtypes = [_f, _f, C.c_float]
        L.l5_forward_out.argtypes = [_f, _f, _f]
        _l5 = L
    return _l5


def l5_init_params(seed=1):
    p = np.empty(L5_NPARAM, np.float32)
    lenet5().l5_init_params(fp(p), seed)
    return p


def l5_batch_grad(p, imgs_f32, labels):
    """sum over the batch of the packed (negative) gradient (float64) and the sum of error norms"""
    imgs = np.ascontiguousarray(imgs_f32, np.float32).reshape(-1, 784)
    labs = np.ascontiguousarray(labels, np.uint8)
    g = np.zeros(L5_NPARAM, np.float64)
    e = np.zeros(1, np.float64)
    lenet5().l5_batch_grad(fp(np.ascontiguousarray(p, np.float32)), fp(imgs.reshape(-1)), u8p(labs), imgs.shape[0], dp(g), dp(e))
    return g, float(e[0])


def l5_apply_update(p, g_f32, step):
    q = np.array(p, np.float32, copy=True)
    lenet5().l5_apply_update(fp(q), fp(np.ascontiguousarray(g_f32, np.float32)), np.float32(step))
    return q


def l5_forward_out(p, img_f32):
    out = np.empty(10, np.float32)
    lenet5().l5_forward_out(fp(np.ascontiguousarray(p, np.float32)), fp(np.ascontiguousarray(img_f32, np.float32).reshape(-1)), fp(out))
    return out


# ---------------------------------------------------------------- convenience wrappers over the oracle
def init_params():
    p = np.empty(NPARAM, np.float32)
    oracle().orc_init_params(fp(p))
    return p


def u8_to_f32(u8):
    u8 = np.ascontiguousarray(u8, np.uint8)
    out = np.empty(u8.shape, np.float32)
    oracle().orc_u8_to_f32(u8p(u8.reshape(-1)), fp(out.reshape(-1)), u8.size)
    return out


def forward(params, img_f32):
    acts = np.empty(N_ACTS, np.float32)
    oracle().orc_forward(fp(params), fp(np.ascontiguousarray(img_f32.reshape(-1))), acts.ctypes.data)
    return acts


def backward(params, img_f32, label, acts):
    back = np.empty(N_BACK, np.float32)
    oracle().orc_backward(fp(params), fp(np.ascontiguousarray(img_f32.reshape(-1))), int(label),
                          acts.ctypes.data, back.ctypes.data)
    return back


def batch_grad(params, imgs_f32, labels_u8):
    """Frozen-weight accumulation (double) of the packed gradient over a batch; returns (g[2343] f64, err_sum)."""
    imgs = np.ascontiguousarray(imgs_f32.reshape(-1, 784), np.float32)
    labels = np.ascontiguousarray(labels_u8, np.uint8)
    g = np.zeros(NPARAM, np.float64)
    es = np.zeros(1, np.float64)
    oracle().orc_batch_grad(fp(params), fp(imgs.reshape(-1)), u8p(labels), imgs.shape[0], dp(g), dp(es))
    return g, float(es[0])


def apply_update(params, g_f32, lr):
    p = params.copy()
    oracle().orc_apply_update(fp(p), fp(np.ascontiguousarray(g_f32, np.float32)), C.c_float(lr))
    return p


def fnv1a32(arr):
    h = 0x811C9DC5
    for b in np.ascontiguousarray(arr).view(np.uint8).tobytes():
        h = ((h ^ b) * 0x01000193) & 0xFFFFFFFF
    return h


def read_idx_images(path):
    raw = np.fromfile(path, np.uint8)
    assert int.from_bytes(raw[0:4].tobytes(), "big") == 2051
    n = int.from_bytes(raw[4:8].tobytes(), "big")
    return raw[16:16 + n * 784].reshape(n, 784).copy()


def read_idx_labels(path):
    raw = np.fromfile(path, np.uint8)
    assert int.from_bytes(raw[0:4].tobytes(), "big") == 2049
    n = int.from_bytes(raw[4:8].tobytes(), "big")
    return raw[8:8 + n].copy()


def full_mnist():
    """(train_images u8 [60000,784], train_labels u8, test_images, test_labels) or None if not staged."""
    f = [os.path.join(REF_DATA, n) for n in ("train-images.idx3-ubyte", "train-labels.idx1-ubyte",
                                             "t10k-images.idx3-ubyte", "t10k-labels.idx1-ubyte")]
    if not all(os.path.exists(x) for x in f):
        return None
    return read_idx_images(f[0]), read_idx_labels(f[1]), read_idx_images(f[2]), read_idx_labels(f[3])


# ---------------------------------------------------------------- stand-ins for the reference's runs on the full dataset
EPOCH_STEPS = 60000     # one epoch of Main.cpp's learn() at batch 1 on the MNIST training split


def fixture_splits(subset):
    """The stored MNIST samples (tests/golden/mnist_subset.npz) shaped like the reference's run: a 60,000-sample training
    split made of the 1,024 stored training samples repeated in order, and the 256 stored test samples as the test split."""
    tr = np.resize(subset["train_u8"], (EPOCH_STEPS, 784))
    trl = np.resize(subset["train_labels"], EPOCH_STEPS)
    return tr, trl, np.ascontiguousarray(subset["test_u8"]), np.ascontiguousarray(subset["test_labels"])


def write_idx(directory, images, labels, stem):
    """`stem`-images.idx3-ubyte and `stem`-labels.idx1-ubyte in the MNIST IDX format mnist.h reads."""
    os.makedirs(directory, exist_ok=True)
    with open(os.path.join(directory, f"{stem}-images.idx3-ubyte"), "wb") as f:
        f.write(np.array([2051, len(images), 28, 28], ">u4").tobytes())
        f.write(np.ascontiguousarray(images, np.uint8).tobytes())
    with open(os.path.join(directory, f"{stem}-labels.idx1-ubyte"), "wb") as f:
        f.write(np.array([2049, len(labels)], ">u4").tobytes())
        f.write(np.ascontiguousarray(labels, np.uint8).tobytes())


def write_fixture_data(directory, subset):
    """The four IDX files Main.cpp's loaddata() opens, holding fixture_splits(subset)."""
    tr, trl, te, tel = fixture_splits(subset)
    write_idx(directory, tr, trl, "train")
    write_idx(directory, te, tel, "t10k")
    return directory


REF_EPOCH = os.path.join(GOLDEN, "reference_fixture_epoch.npz")
REF_OPS = os.path.join(GOLDEN, "reference_ops.json")


def reference_fixture_epoch():
    """What the reference computed on fixture_splits() (oracle/gen_golden.py): its driver's printed lines, the mean error of
    the epoch, the mismatches of its test() and its parameters after the epoch."""
    return dict(np.load(REF_EPOCH))


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a, np.float32).tobytes()).hexdigest()


# the reference's spelling where the oracle's entry point is named differently
_REF_OP_NAMES = {"make_error": "makeError", "vector_norm": "vectorNorm"}


def op_chain(L, prefix, rng, label):
    """Every layer.h operator once, on inputs drawn from `rng`, each fed with the outputs of the ones before it as Main.cpp's
    forward and backward passes feed them.  L is the oracle (prefix "orc_") or the compiled reference ("ref_").  Returns
    [(name, float32 array)] in call order, the drawn inputs first."""
    def op(name, *args):
        return getattr(L, prefix + (_REF_OP_NAMES.get(name, name) if prefix == "ref_" else name))(*args)

    def r(*shape, lo=-1.0, hi=1.0):
        return np.ascontiguousarray(rng.uniform(lo, hi, shape).astype(np.float32))

    inp, w1, b1 = r(784, lo=0, hi=1), r(150, lo=-.5, hi=.5), r(6, lo=-.5, hi=.5)
    w2, b2 = r(16), r(1)
    x216, wf, bf = r(216, lo=0, hi=1), r(2160), r(10)
    out10 = r(10, lo=0, hi=1)
    z = lambda n: np.zeros(n, np.float32)  # noqa: E731
    o1, s1, p1, f1, e1 = z(3456), z(3456), z(216), z(10), z(10)
    op("fp_c1", fp(inp), fp(o1), fp(w1), fp(b1))
    op("apply_step_function", fp(o1), fp(s1), 3456)
    op("fp_s1", fp(s1), fp(p1), fp(w2), fp(b2))
    op("fp_preact_f", fp(x216), fp(f1), fp(wf))
    op("fp_bias_f", fp(f1), fp(bf))
    op("make_error", fp(e1), fp(out10), label, 10)
    norm = np.array([op("vector_norm", fp(e1), 10)], np.float32)
    d1, q1, t1, g1, u1, v1, h1 = z(2160), z(216), z(216), z(16), z(3456), z(3456), z(150)
    bfa, b2a, b1a, wfa = bf.copy(), b2.copy(), b1.copy(), wf.copy()
    op("bp_weight_f", fp(d1), fp(e1), fp(x216))
    op("bp_bias_f", fp(bfa), fp(e1))
    op("bp_output_s1", fp(q1), fp(wf), fp(e1))
    op("bp_preact_s1", fp(t1), fp(q1), fp(p1))
    op("bp_weight_s1", fp(g1), fp(t1), fp(s1))
    op("bp_bias_s1", fp(b2a), fp(t1))
    op("bp_output_c1", fp(u1), fp(w2), fp(t1))
    op("bp_preact_c1", fp(v1), fp(u1), fp(o1))
    op("bp_weight_c1", fp(h1), fp(v1), fp(inp))
    op("bp_bias_c1", fp(b1a), fp(v1))
    op("apply_grad", fp(wfa), fp(d1), 2160)
    inputs = np.concatenate([inp, w1, b1, w2, b2, x216, wf, bf, out10])
    return [("inputs", inputs), ("fp_c1", o1), ("apply_step_function", s1), ("fp_s1", p1), ("fp_preact_f + fp_bias_f", f1),
            ("makeError", e1), ("vectorNorm", norm), ("bp_weight_f", d1), ("bp_bias_f", bfa), ("bp_output_s1", q1),
            ("bp_preact_s1", t1), ("bp_weight_s1", g1), ("bp_bias_s1", b2a), ("bp_output_c1", u1), ("bp_preact_c1", v1),
            ("bp_weight_c1", h1), ("bp_bias_c1", b1a), ("apply_grad", wfa)]
