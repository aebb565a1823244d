"""CPU tests (no GPU): the oracle is pinned to the reference.

1. oracle/liblenet_oracle.so (C restatement) reproduces, bit for bit, the golden vectors that oracle/gen_golden.py
   recorded from the UNMODIFIED reference (tests/golden/reference_vectors.npz) and the SURVEY.md Appendix B scalars.
2. Every operator of the restatement is also compared bit for bit with the reference's own function on random inputs,
   through the output digests oracle/gen_golden.py recorded from the reference (tests/golden/reference_ops.json).
"""
import json

import numpy as np
import pytest

import oracle_lib as O


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def test_init_params_match_reference_constructor(golden):
    p = O.init_params()
    assert np.array_equal(bits(p), bits(golden["params_init"]))
    sc = golden["scalars"]
    assert "%08x" % O.fnv1a32(p[0:150]) == sc["init.fnv.c1w"] == "590b0358"      # SURVEY.md Appendix B
    assert "%08x" % O.fnv1a32(p[173:2333]) == sc["init.fnv.fw"] == "9548d81a"
    assert abs(float(p[150]) - (-0.340187728)) < 1e-9 and abs(float(p[172]) - 0.430093586) < 1e-9


def test_forward_matches_reference_first8(golden):
    p = golden["params_init"]
    for s in range(8):
        a = O.forward(p, O.u8_to_f32(golden["train_u8"][s]))
        assert np.array_equal(bits(a), bits(golden["acts_init_first8"][s])), f"sample {s}"
    # Appendix B: f.out of sample 0
    f_out = O.forward(p, O.u8_to_f32(golden["train_u8"][0]))[7354:]
    np.testing.assert_allclose(f_out[:3], [0.0462899208, 0.0214242004, 0.890034854], rtol=0, atol=1e-9)


def test_step1_backward_buffers_match_reference(golden):
    p = golden["params_init"]
    img = O.u8_to_f32(golden["train_u8"][0])
    lab = int(golden["train_labels"][0])
    a = O.forward(p, img)
    b = O.backward(p, img, lab, a)
    ref = golden["back_step1"]   # f.d_preact, s1.d_output, s1.d_preact, c1.d_output, c1.d_preact, c1.dW, s1.dW, f.dW
    for name, (lo, hi), (rlo, rhi) in [("f_dpre", O.BACK_OFF["f_dpre"], (0, 10)), ("s1_dout", O.BACK_OFF["s1_dout"], (10, 226)),
                                       ("s1_dpre", O.BACK_OFF["s1_dpre"], (226, 442)), ("c1_dout", O.BACK_OFF["c1_dout"], (442, 3898)),
                                       ("c1_dpre", O.BACK_OFF["c1_dpre"], (3898, 7354))]:
        assert np.array_equal(bits(b[lo:hi]), bits(ref[rlo:rhi])), name
    g = b[slice(*O.BACK_OFF["g"])]
    assert np.array_equal(bits(g[0:150]), bits(ref[7354:7504]))          # c1.d_weight
    assert np.array_equal(bits(g[156:172]), bits(ref[7504:7520]))        # s1.d_weight
    assert np.array_equal(bits(g[173:2333]), bits(ref[7520:9680]))       # f.d_weight
    assert float(b[O.BACK_OFF["err"][0]]) == golden["scalars"]["sample0.err"]
    # the update (bias blocks included) lands exactly on the reference's post-step parameters
    p1 = O.apply_update(p, g, 0.1)
    assert np.array_equal(bits(p1), bits(golden["params_after1"]))


def test_trajectory_1000_steps_bit_exact(golden):
    p = golden["params_init"].copy()
    orc = O.oracle()
    errs = np.empty(1000, np.float32)
    for s in range(1000):
        errs[s] = orc.orc_train_step(O.fp(p), O.fp(O.u8_to_f32(golden["train_u8"][s])), int(golden["train_labels"][s]))
    assert np.array_equal(bits(errs), bits(golden["err_first1000"]))
    assert np.array_equal(bits(p), bits(golden["params_after1000"]))
    assert "%08x" % O.fnv1a32(p[0:150]) == "996f4aa7" and "%08x" % O.fnv1a32(p[173:2333]) == "c79d0029"   # Appendix B
    # classify() on the test subset
    pred = np.array([orc.orc_classify(O.fp(p), O.fp(O.u8_to_f32(golden["test_u8"][s]))) for s in range(256)], np.uint8)
    assert np.array_equal(pred, golden["pred_test_sub_after1000"])
    wrong = orc.orc_test(O.fp(p), O.u8p(golden["test_u8"].reshape(-1)), O.u8p(golden["test_labels"]), 256)
    assert wrong == int(golden["wrong_test_sub_after1000"])


def test_learn_loop_matches_on_subset(golden):
    p = golden["params_init"].copy()
    e = O.oracle().orc_learn(O.fp(p), O.u8p(golden["train_u8"].reshape(-1)), O.u8p(golden["train_labels"]), 1000)
    acc = np.float32(0)
    for v in golden["err_first1000"]:
        acc = np.float32(acc + v)                      # Main.cpp:169 fp32 running sum
    assert e == np.float32(acc / np.float32(1000))


def test_batch_oracle_is_sum_of_per_sample_gradients(golden):
    p = golden["params_init"]
    imgs = O.u8_to_f32(golden["train_u8"][:5])
    labs = golden["train_labels"][:5]
    g, es = O.batch_grad(p, imgs, labs)
    acc = np.zeros(O.NPARAM, np.float64)
    e2 = 0.0
    for s in range(5):
        a = O.forward(p, imgs[s])
        b = O.backward(p, imgs[s], int(labs[s]), a)
        acc += b[slice(*O.BACK_OFF["g"])].astype(np.float64)
        e2 += float(b[O.BACK_OFF["err"][0]])
    assert np.array_equal(g, acc) and es == e2


def test_pixel_conversion_single_division_equals_double_route():
    # the CUDA kernels convert with one fp32 division; mnist.h:145 + Main.cpp:64 go through double
    u = np.arange(256, dtype=np.uint8)
    assert np.array_equal(bits(O.u8_to_f32(u)), bits(u.astype(np.float32) / np.float32(255.0)))


# --------------------------------------------------------------------------- comparison with the reference's own functions
@pytest.fixture(scope="module")
def ref_ops():
    with open(O.REF_OPS) as f:
        return json.load(f)


def test_ops_bit_exact_vs_reference_on_random_inputs(ref_ops):
    """Every operator of the restatement against the reference's own function on the same random inputs: the SHA-256 of
    each output's bits equals the one oracle/gen_golden.py recorded from the reference (tests/golden/reference_ops.json)."""
    rng = np.random.default_rng(ref_ops["seed"])
    for trial, ref in enumerate(ref_ops["trials"]):
        got = O.op_chain(O.oracle(), "orc_", rng, trial)
        assert [name for name, _ in got] == list(ref)
        for name, a in got:
            assert O.digest(a) == ref[name], f"trial {trial}: {name}"


def test_reference_static_constructor_state_equals_seed1_redraw(golden, ref_ops):
    """The reference's parameters after srand(1) and a redraw in constructor order are its static-constructor state."""
    assert ref_ops["params_static_constructors"] == ref_ops["params_after_reset"] == O.digest(golden["params_init"])
    assert ref_ops["sizeof_mnist_data"] == 6280            # Appendix B


def test_lenet5_variant_oracle_backward_is_the_gradient_of_its_forward(golden):
    """oracle/lenet5_oracle.c is self-written (the reference has no second conv layer): its backward pass is pinned to its
    own forward pass by a finite-difference check.  With d_preact_f = onehot - output (layer.h:91-95) the packed vector is
    the negative gradient of the summed binary cross-entropy of the ten sigmoid outputs, up to the normalisation rules
    (conv weight blocks divided by the map size: 576 for c1, 64 for c3)."""
    p0 = O.l5_init_params(7).astype(np.float64)
    img = O.u8_to_f32(golden["train_u8"][3])
    y = int(golden["train_labels"][3])
    t = np.zeros(10)
    t[y] = 1.0

    def loss(pv):
        o = O.l5_forward_out(pv.astype(np.float32), img).astype(np.float64)
        return -np.sum(t * np.log(o) + (1 - t) * np.log(1 - o))

    g, err = O.l5_batch_grad(p0.astype(np.float32), img[None], np.array([y], np.uint8))
    assert np.isfinite(g).all() and err > 0
    scale = np.ones(O.L5_NPARAM)
    scale[slice(*O.L5_OFF["c1w"])] = 576.0
    scale[slice(*O.L5_OFF["c3w"])] = 64.0
    rng = np.random.default_rng(0)
    picks = np.concatenate([rng.choice(np.arange(*O.L5_OFF[k]), size=min(6, O.L5_OFF[k][1] - O.L5_OFF[k][0]), replace=False)
                            for k in O.L5_OFF])
    for j in picks:
        eps = 2e-2
        pp, pm = p0.copy(), p0.copy()
        pp[j] += eps
        pm[j] -= eps
        num = -(loss(pp) - loss(pm)) / (2 * eps)            # negative gradient, like the packed vector
        ana = g[j] * scale[j]
        assert abs(num - ana) <= 3e-2 * max(abs(ana), abs(num)) + 2e-4, (int(j), num, ana)
