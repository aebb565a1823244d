"""GPU test of the reference-shaped C++ driver (parallel-cnn_b200/driver/main.cpp) built on include/layer.h.

The drivers read the four IDX files of O.fixture_splits (the stored MNIST samples shaped as the reference's 60,000-step
epoch) and are compared with what the reference computed on the same files (tests/golden/reference_fixture_epoch.npz)."""
import os
import re
import subprocess

import numpy as np
import pytest

import oracle_lib as O

pytestmark = pytest.mark.gpu
DRIVER = os.path.join(O.ROOT, "parallel-cnn_b200", "driver", "pcnn_main")


@pytest.fixture(scope="module")
def data_dir(tmp_path_factory, golden):
    return O.write_fixture_data(str(tmp_path_factory.mktemp("mnist") / "data"), golden)


@pytest.fixture(scope="module")
def ref_epoch():
    return O.reference_fixture_epoch()


def run(data_dir, *args):
    r = subprocess.run([DRIVER, "--data", data_dir, *args], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    return r.stdout


def test_driver_default_replays_the_reference_run(data_dir, ref_epoch):
    out = run(data_dir)                               # batch 1, 1 epoch: Sequential/Main.cpp's own run
    assert out.startswith("Learning\n")
    err = float(re.search(r"error: ([0-9.e+-]+), time_on_cpu", out).group(1))
    rate = float(re.search(r"Error Rate: ([0-9.]+)%", out).group(1))
    assert abs(err - float(ref_epoch["epoch_err"])) <= 2e-3, err
    assert abs(rate - float(ref_epoch["rate_printed"])) <= 0.3, rate
    for line in ("Total Convolution Time:", "Total Pooling Time:", "Total Fully Connected Time:",
                 "Total Time on applying gradients:", " Time - "):
        assert line in out


def test_driver_operator_mode_matches_reference_errors(data_dir, golden):
    out = run(data_dir, "--ops", "--limit", "200")    # the 18 layer.h functions called in Main.cpp's order, per sample
    err = float(re.search(r"error: ([0-9.e+-]+), time_on_cpu", out).group(1))
    ref = float(golden["err_first1000"][:200].astype(np.float64).mean())
    assert abs(err - ref) <= 1e-4 * ref
    rate = float(re.search(r"Error Rate: ([0-9.]+)%", out).group(1))
    assert 0.0 <= rate <= 100.0


def test_driver_reports_missing_data_like_mnist_load():
    r = subprocess.run([DRIVER, "--data", "/nonexistent"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 1 and "mnist_load code -1" in r.stderr


DROPIN = os.path.join(O.ROOT, "oracle", "_ref", "seq_main_b200")


@pytest.mark.skipif(not os.path.exists(DROPIN),
                    reason="oracle/_ref/seq_main_b200 is compiled from the reference's own sources, only where they exist "
                           "(oracle/Makefile: dropin)")
def test_the_reference_driver_itself_runs_on_the_engine(data_dir, ref_epoch):
    """INTEGRATION.md section 1, literally: the reference's own Sequential/Main.cpp, with only its two host dereferences of
    device memory rewritten (Main.cpp:168, :191), compiled against include/layer.h and linked to libpcnn.so.  Every one of
    its 60,000 x 18 operator calls and its classify() calls goes through the C ABI (operator tier: reference operation
    order, double-precision sigmoid), so its two printed results are the reference's own."""
    r = subprocess.run([DROPIN], cwd=os.path.dirname(data_dir), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr
    out = r.stdout
    err = float(re.search(r"error: ([0-9.e+-]+), time_on_cpu", out).group(1))
    rate = float(re.search(r"Error Rate: ([0-9.]+)%", out).group(1))
    assert abs(err - float(ref_epoch["epoch_err"])) <= 1e-5
    assert abs(rate - float(ref_epoch["rate_printed"])) <= 0.011
