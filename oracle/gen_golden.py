#!/usr/bin/env python
"""Generate tests/golden/ from the UNMODIFIED reference (oracle/_ref/libref_seq.so).

TEST INFRASTRUCTURE ONLY.  Run in the authoring container (needs /root/reference to have been compiled by
`make -C oracle`).  The reference ships no tests or golden vectors (SURVEY.md section 4), so every fixture is an
output of the reference's own code on real MNIST bytes:

  mnist_subset.npz       first 1024 training and first 256 test samples, raw u8 + labels (the IDX payload bytes)
  reference_vectors.npz  seed-1 parameters, per-sample activations / backward buffers, parameter states after
                         1, 1000 and 60000 steps, per-step error norms, classifications
  reference_scalars.json the SURVEY.md Appendix B numbers re-measured here (err, error rate, sums, FNV hashes)
  reference_ops.json     SHA-256 of every operator output of the reference on seeded random inputs, and of its
                         parameters after the seed-1 redraw
  reference_fixture_epoch.npz  the reference's own driver and learn loop on the stored samples shaped as a full epoch
                         (oracle_lib.fixture_splits): printed lines, mean error, test mismatches, final parameters
The last two let the tests compare with the reference where it cannot be built; `--selfcontained` writes only them.
"""
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tests"))
import oracle_lib as O  # noqa: E402

N_TRAIN_SUB, N_TEST_SUB = 1024, 256


def main():
    ref = O.reference()
    if ref is None:
        raise SystemExit("oracle/_ref/libref_seq.so missing: run `make -C oracle` where /root/reference exists")
    data = O.full_mnist()
    if data is None:
        raise SystemExit("oracle/_ref/data missing")
    tr, trl, te, tel = data
    os.makedirs(O.GOLDEN, exist_ok=True)
    np.savez_compressed(os.path.join(O.GOLDEN, "mnist_subset.npz"),
                        train_u8=tr[:N_TRAIN_SUB], train_labels=trl[:N_TRAIN_SUB],
                        test_u8=te[:N_TEST_SUB], test_labels=tel[:N_TEST_SUB])

    def params():
        p = np.empty(O.NPARAM, np.float32)
        ref.ref_get_params(O.fp(p))
        return p

    def acts():
        a = np.empty(O.N_ACTS, np.float32)
        ref.ref_get_acts(O.fp(a))
        return a

    def back():
        b = np.empty(7520 + 2160, np.float32)
        ref.ref_get_back(O.fp(b))
        return b

    out = {}
    sc = {}
    ref.ref_reset_params()
    p0 = params()
    out["params_init"] = p0
    # forward records for the first 8 samples with the seed-1 parameters
    fa = []
    for s in range(8):
        ref.ref_forward_u8(O.u8p(tr[s]))
        fa.append(acts())
    out["acts_init_first8"] = np.stack(fa)
    # step-by-step: backward record of step 1, error norms of the first 1000 steps
    errs = np.empty(1000, np.float32)
    for s in range(1000):
        errs[s] = ref.ref_train_step_u8(O.u8p(tr[s]), int(trl[s]))
        if s == 0:
            out["back_step1"] = back()
            out["acts_step1"] = acts()
            out["params_after1"] = params()
    out["err_first1000"] = errs
    out["params_after1000"] = params()
    out["pred_test_sub_after1000"] = np.array([ref.ref_classify_u8(O.u8p(te[s])) for s in range(N_TEST_SUB)], np.uint8)
    out["wrong_test_sub_after1000"] = np.array(ref.ref_test_u8(O.u8p(te[:N_TEST_SUB].reshape(-1)), O.u8p(tel[:N_TEST_SUB]), N_TEST_SUB))
    # continue to 20,000 then a full epoch from scratch through the driver-shaped loop
    ref.ref_reset_params()
    secs = np.zeros(1, np.float64)
    e20k = ref.ref_learn_loop_u8(O.u8p(tr[:20000].reshape(-1)), O.u8p(trl[:20000]), 20000, O.dp(secs))
    sc["mean_err_first_20000"] = float(e20k)
    ref.ref_reset_params()
    e_epoch = ref.ref_learn_loop_u8(O.u8p(tr.reshape(-1)), O.u8p(trl), 60000, O.dp(secs))
    sc["epoch_err"] = float(e_epoch)
    sc["epoch_err_printed"] = "%e" % e_epoch
    sc["epoch_seconds_here"] = float(secs[0])
    out["params_after_epoch"] = params()
    wrong = int(ref.ref_test_u8(O.u8p(te.reshape(-1)), O.u8p(tel), 10000))
    sc["test_wrong_after_epoch"] = wrong
    sc["test_error_rate_printed"] = "%.2lf%%" % (wrong / 10000.0 * 100.0)
    out["pred_test_sub_after_epoch"] = np.array([ref.ref_classify_u8(O.u8p(te[s])) for s in range(N_TEST_SUB)], np.uint8)

    def sums(p, tag):
        for k, (a, b) in O.OFF.items():
            sc[f"{tag}.sum.{k}"] = float(np.sum(p[a:b].astype(np.float64)))
        sc[f"{tag}.fnv.c1w"] = "%08x" % O.fnv1a32(p[0:150])
        sc[f"{tag}.fnv.fw"] = "%08x" % O.fnv1a32(p[173:2333])

    sums(p0, "init")
    sums(out["params_after1"], "after1")
    sums(out["params_after1000"], "after1000")
    sums(out["params_after_epoch"], "after_epoch")
    sc["sample0.err"] = float(errs[0])
    sc["sizeof_mnist_data"] = int(ref.ref_sizeof_mnist_data())
    np.savez_compressed(os.path.join(O.GOLDEN, "reference_vectors.npz"), **out)
    with open(os.path.join(O.GOLDEN, "reference_scalars.json"), "w") as f:
        json.dump(sc, f, indent=1, sort_keys=True)
    print(json.dumps(sc, indent=1, sort_keys=True))


OPS_TRIALS, OPS_SEED = 5, 1234


def selfcontained():
    """Must run on a freshly loaded reference: its first record is the static constructors' parameter state."""
    ref = O.reference()
    if ref is None:
        raise SystemExit("oracle/_ref/libref_seq.so missing: run `make -C oracle` where the reference sources exist")
    p = np.empty(O.NPARAM, np.float32)
    ref.ref_get_params(O.fp(p))
    static = O.digest(p)
    rng = np.random.default_rng(OPS_SEED)
    trials = [{name: O.digest(a) for name, a in O.op_chain(ref, "ref_", rng, t)} for t in range(OPS_TRIALS)]
    ref.ref_reset_params()
    ref.ref_get_params(O.fp(p))
    ops = {"seed": OPS_SEED, "trials": trials, "params_static_constructors": static, "params_after_reset": O.digest(p),
           "sizeof_mnist_data": int(ref.ref_sizeof_mnist_data())}
    with open(O.REF_OPS, "w") as f:
        json.dump(ops, f, indent=1)

    subset = np.load(os.path.join(O.GOLDEN, "mnist_subset.npz"))
    tr, trl, te, tel = O.fixture_splits(subset)
    ref.ref_reset_params()
    secs = np.zeros(1, np.float64)
    err = ref.ref_learn_loop_u8(O.u8p(tr.reshape(-1)), O.u8p(trl), len(trl), O.dp(secs))
    ref.ref_get_params(O.fp(p))
    wrong = int(ref.ref_test_u8(O.u8p(te.reshape(-1)), O.u8p(tel), len(tel)))
    # the reference's own driver (Sequential/Main.cpp, unmodified) on the same four files prints the same two results
    with tempfile.TemporaryDirectory() as tmp:
        O.write_fixture_data(os.path.join(tmp, "data"), subset)
        out = subprocess.run([os.path.join(O.ROOT, "oracle", "_ref", "seq_main")], cwd=tmp, capture_output=True, text=True,
                             check=True).stdout
    err_printed = re.search(r"error: (\S+), time_on_cpu", out).group(1)
    rate_printed = re.search(r"Error Rate: (\S+)%", out).group(1)
    assert err_printed == "%e" % err and rate_printed == "%.2f" % (wrong / len(tel) * 100.0), (out, err, wrong)
    np.savez_compressed(O.REF_EPOCH, epoch_err=np.float32(err), test_wrong=np.int64(wrong), test_count=np.int64(len(tel)),
                        err_printed=np.array(err_printed), rate_printed=np.array(rate_printed), params_after_epoch=p)
    print(json.dumps({"epoch_err": float(err), "err_printed": err_printed, "test_wrong": wrong, "rate_printed": rate_printed}))


if __name__ == "__main__":
    selfcontained()
    if "--selfcontained" not in sys.argv[1:]:
        main()
