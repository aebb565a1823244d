"""GPU parity tests of the fused training / evaluation path (the fast tier) through the C ABI.

Tolerances (DESIGN.md "numerics"; SURVEY.md 8c protocol).  The fused kernels use FMA, tree-ordered sums and a float
sigmoid, so they are not bit-exact; the stated bounds are
  op level     |d| <= 1e-6 + 1e-5 |ref|                 (f.output per sample)
  step level   rel-L2(packed gradient) <= 1e-5 vs the frozen-weight oracle sum, B in {1, 7, 256, 1024}
  trajectory   rel-L2(parameters) <= 1e-3 after the first 1000 B=1 steps vs the reference's recorded state
  epoch        mean err within 2e-3, test error rate within 0.3 pp of the reference's on the same 60,000-step epoch
Size-independent properties cover the BASELINE batch sizes the oracle would take too long for (8192): run-to-run
determinism (bit-identical), u8/f32 input equivalence, additivity of the batch gradient.
"""
import os

import numpy as np
import pytest

import oracle_lib as O

pytestmark = pytest.mark.gpu


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


@pytest.fixture(scope="module")
def data(eng, golden, pkg):
    d = dict(train=golden["train_u8"], labels=golden["train_labels"], test=golden["test_u8"], test_labels=golden["test_labels"])
    d["train_f32"] = O.u8_to_f32(d["train"])
    d["d_train"] = eng.to_device(d["train"])
    d["d_train_f32"] = eng.to_device(d["train_f32"])
    d["d_labels"] = eng.to_device(d["labels"])
    d["d_test"] = eng.to_device(d["test"])
    return d


@pytest.mark.parametrize("B", [1, 7, 256, 1024])
def test_step_gradient_vs_frozen_weight_oracle(eng, pkg, golden, data, B):
    p = golden["params_init"]
    eng.set_params(p)
    eng.compute_grads(data["d_train"], pkg.U8, data["d_labels"], B)
    g = eng.get_grads()
    g_ref, err_ref = O.batch_grad(p, data["train_f32"][:B], data["labels"][:B])
    assert rel_l2(g, g_ref) <= 1e-5
    for name, (lo, hi) in O.OFF.items():                     # every block on its own, too
        assert rel_l2(g[lo:hi], g_ref[lo:hi]) <= 2e-5, name
    assert np.array_equal(eng.get_params().view(np.uint32), p.view(np.uint32))      # compute_grads must not update


def test_u8_and_f32_inputs_are_equivalent(eng, pkg, golden, data):
    eng.set_params(golden["params_init"])
    eng.compute_grads(data["d_train"], pkg.U8, data["d_labels"], 300)
    g8 = eng.get_grads()
    eng.compute_grads(data["d_train_f32"], pkg.F32, data["d_labels"], 300)
    g32 = eng.get_grads()
    assert np.array_equal(g8.view(np.uint32), g32.view(np.uint32))


def test_step_is_deterministic_and_additive_at_8192(eng, pkg, golden, data):
    eng.set_params(golden["params_init"])
    big = np.tile(data["train"], (8, 1))                      # 8192 samples = the 1024-sample fixture eight times
    lab = np.tile(data["labels"], 8)
    d_big, d_lab = eng.to_device(big), eng.to_device(lab)
    eng.compute_grads(d_big, pkg.U8, d_lab, 8192)
    g1 = eng.get_grads()
    eng.compute_grads(d_big, pkg.U8, d_lab, 8192)
    g2 = eng.get_grads()
    assert np.array_equal(g1.view(np.uint32), g2.view(np.uint32))                    # no atomics: bit-identical reruns
    eng.compute_grads(data["d_train"], pkg.U8, data["d_labels"], 1024)
    g1024 = eng.get_grads()
    assert rel_l2(g1, 8.0 * g1024.astype(np.float64)) <= 1e-5                        # additivity over the batch


def test_train_step_update_matches_oracle(eng, pkg, golden, data):
    for B in (1, 256):
        p = golden["params_init"]
        eng.set_params(p)
        eng.err_sum(reset=True)
        eng.train_step_dev(data["d_train"], pkg.U8, data["d_labels"], B)
        got = eng.get_params()
        g_ref, err_ref = O.batch_grad(p, data["train_f32"][:B], data["labels"][:B])
        exp = O.apply_update(p, g_ref.astype(np.float32), np.float32(0.1) / np.float32(B))
        np.testing.assert_allclose(got, exp, rtol=2e-6, atol=2e-7)
        assert abs(eng.err_sum() - err_ref) <= 1e-5 * err_ref
    # B = 1 is the reference's own step: compare with the recorded post-step parameters
    eng.set_params(golden["params_init"])
    eng.train_step_dev(data["d_train"], pkg.U8, data["d_labels"], 1)
    np.testing.assert_allclose(eng.get_params(), golden["params_after1"], rtol=2e-6, atol=2e-7)


def test_trajectory_first_1000_reference_steps(eng, pkg, golden, data):
    eng.dataset_upload(pkg.TRAIN_SET, data["train"][:1000], data["labels"][:1000])
    eng.set_params(golden["params_init"])
    eng.err_sum(reset=True)
    eng.train_steps(0, 1, 1000)                        # cursor-driven, graph-replayed B = 1 steps in dataset order
    p = eng.get_params()
    assert rel_l2(p, golden["params_after1000"]) <= 1e-3
    assert abs(eng.err_sum() - float(golden["err_first1000"].astype(np.float64).sum())) <= 1e-3 * 1000 * 0.33
    # learn() over the same split gives the same state (one epoch of 1000 samples) and reports err / n
    eng.set_params(golden["params_init"])
    mean_err = eng.learn(B=1, epochs=1)
    assert np.array_equal(eng.get_params().view(np.uint32), p.view(np.uint32))
    assert abs(mean_err - float(golden["err_first1000"].astype(np.float64).mean())) <= 1e-3


def test_train_step_on_bound_split_and_tail_batch(eng, pkg, golden, data):
    n = 1000
    eng.dataset_upload(pkg.TRAIN_SET, data["train"][:n], data["labels"][:n])
    # explicit window
    eng.set_params(golden["params_init"])
    eng.train_step(512, 256)
    a = eng.get_params()
    eng.set_params(golden["params_init"])
    d_i, d_l = eng.to_device(data["train"][512:768]), eng.to_device(data["labels"][512:768])
    eng.train_step_dev(d_i, pkg.U8, d_l, 256)
    assert np.array_equal(a.view(np.uint32), eng.get_params().view(np.uint32))
    # learn() with a ragged tail: 1000 = 3 * 256 + 232, the last step uses dt / 232
    eng.set_params(golden["params_init"])
    eng.learn(B=256, epochs=1)
    got = eng.get_params()
    p = golden["params_init"]
    for lo in range(0, n, 256):
        hi = min(n, lo + 256)
        g, _ = O.batch_grad(p, data["train_f32"][lo:hi], data["labels"][lo:hi])
        p = O.apply_update(p, g.astype(np.float32), np.float32(0.1) / np.float32(hi - lo))
    np.testing.assert_allclose(got, p, rtol=5e-6, atol=5e-7)
    with pytest.raises(pkg.PcnnError):
        eng.train_step(900, 256)                       # window past the end of the split


def test_host_entry_points_match_device_path(eng, pkg, golden, data):
    n, B = 1000, 128
    eng.dataset_upload(pkg.TRAIN_SET, data["train"][:n], data["labels"][:n])
    eng.set_params(golden["params_init"])
    e_dev = eng.learn(B=B, epochs=1)
    p_dev = eng.get_params()
    eng.set_params(golden["params_init"])
    e_host = eng.learn_host(data["train"][:n], data["labels"][:n], B=B, epochs=1)
    assert np.array_equal(p_dev.view(np.uint32), eng.get_params().view(np.uint32))
    assert abs(e_dev - e_host) < 1e-6
    eng.set_params(golden["params_init"])
    e = eng.train_step_host(data["train"][:B], data["labels"][:B])
    _, err_ref = O.batch_grad(golden["params_init"], data["train_f32"][:B], data["labels"][:B])
    assert abs(e - err_ref) <= 1e-5 * err_ref


@pytest.mark.parametrize("B,n", [(128, 1000), (1, 37), (256, 1024), (512, 900)])
def test_pinned_host_images_are_pulled_by_the_kernel_and_match_the_staged_path(eng, pkg, golden, data, B, n):
    """pcnn_learn_host with page-locked images: the training kernel reads them across PCIe itself (no staging copy); pageable
    images go through the staged copy stream.  Same samples, same order -> bit-identical parameters and per-step errors, also
    against the device-resident path; two epochs re-read the host buffer."""
    import torch
    imgs, labs = data["train"][:n], data["labels"][:n]
    eng.dataset_upload(pkg.TRAIN_SET, imgs, labs)
    eng.set_params(golden["params_init"])
    e_dev = eng.learn(B=B, epochs=2)
    p_dev = eng.get_params()
    hi = torch.empty((n, 784), dtype=torch.uint8, pin_memory=True)
    hl = torch.empty((n,), dtype=torch.uint8, pin_memory=True)
    hi.numpy()[:] = imgs
    hl.numpy()[:] = labs
    eng.set_params(golden["params_init"])
    e_pull = eng.learn_host(hi.numpy(), hl.numpy(), B=B, epochs=2)
    errs_pull = eng.step_errs().copy()
    assert np.array_equal(p_dev.view(np.uint32), eng.get_params().view(np.uint32))
    assert abs(e_dev - e_pull) < 1e-6
    eng.set_params(golden["params_init"])
    e_staged = eng.learn_host(np.array(imgs, copy=True), np.array(labs, copy=True), B=B, epochs=2)     # pageable
    assert np.array_equal(p_dev.view(np.uint32), eng.get_params().view(np.uint32))
    assert np.array_equal(errs_pull.view(np.uint32), eng.step_errs().view(np.uint32)) and abs(e_pull - e_staged) < 1e-6
    eng.persist_tune(16)                                # pinned memory through the staged stream (the A/B knob)
    try:
        eng.set_params(golden["params_init"])
        eng.learn_host(hi.numpy(), hl.numpy(), B=B, epochs=2)
        assert np.array_equal(p_dev.view(np.uint32), eng.get_params().view(np.uint32))
    finally:
        eng.persist_tune(0)
    # fp32 pixels, pinned
    hf = torch.empty((n, 784), dtype=torch.float32, pin_memory=True)
    hf.numpy()[:] = data["train_f32"][:n]
    eng.set_params(golden["params_init"])
    eng.learn_host(hf.numpy(), hl.numpy(), B=B, epochs=2)
    assert np.array_equal(p_dev.view(np.uint32), eng.get_params().view(np.uint32))


def test_forward_batch_and_classify(eng, pkg, golden, data):
    p = golden["params_after1000"]
    eng.set_params(p)
    B = 256
    f_out, pred = eng.array((B, 10)), eng.array(B, np.uint8)
    eng.forward_batch(data["d_test"], pkg.U8, B, f_out, pred)
    ref = np.stack([O.forward(p, O.u8_to_f32(data["test"][s]))[7354:] for s in range(B)])
    got = f_out.to_host()
    assert np.all(np.abs(got - ref) <= 1e-6 + 1e-5 * np.abs(ref))
    assert np.array_equal(pred.to_host(), golden["pred_test_sub_after1000"])       # first-max argmax, Main.cpp:193-197
    eng.dataset_upload(pkg.TEST_SET, data["test"], data["test_labels"])
    assert eng.test() == int(golden["wrong_test_sub_after1000"])


def test_checkpoint_roundtrip(eng, golden, tmp_path):
    eng.set_params(golden["params_after1000"])
    path = str(tmp_path / "w.pcnn")
    eng.save_params(path)
    assert os.path.getsize(path) == 16 + 9372
    eng.set_params(golden["params_init"])
    eng.load_params(path)
    assert np.array_equal(eng.get_params().view(np.uint32), golden["params_after1000"].view(np.uint32))


def test_fused_argument_errors(eng, pkg, data):
    with pytest.raises(pkg.PcnnError) as ei:
        eng.compute_grads(data["d_train"], pkg.U8, data["d_labels"], 0)
    assert ei.value.code == -1
    with pytest.raises(pkg.PcnnError):
        eng.compute_grads(data["d_train"].ptr + 4, pkg.U8, data["d_labels"], 4)      # bulk-copy source must be 16-B aligned
    with pytest.raises(pkg.PcnnError):
        eng.compute_grads(data["d_train"], 7, data["d_labels"], 4)


def test_full_epoch_reproduces_reference_headline(eng, pkg, golden):
    """Config 1 of BASELINE.json: the whole of Main.cpp (learn + test) at batch 1, one 60,000-step epoch, on the stored
    samples shaped as the reference's run (O.fixture_splits), against the reference's results on the same splits."""
    tr, trl, te, tel = O.fixture_splits(golden)
    ref = O.reference_fixture_epoch()
    eng.dataset_upload(pkg.TRAIN_SET, tr, trl)
    eng.dataset_upload(pkg.TEST_SET, te, tel)
    eng.set_params(golden["params_init"])
    mean_err = eng.learn(B=1, epochs=1)
    wrong = eng.test()
    assert abs(mean_err - float(ref["epoch_err"])) <= 2e-3, mean_err
    assert abs(wrong - int(ref["test_wrong"])) <= 0.003 * len(tel), wrong          # +- 0.3 pp of the test split
    assert rel_l2(eng.get_params(), ref["params_after_epoch"]) <= 5e-2
