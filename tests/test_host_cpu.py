"""CPU tests (no GPU) of the host-side logic and of the C-ABI library as a loadable object.  No compute entry point is
called here: without a GPU pcnn_create must fail loudly (no CPU fallback)."""
import ctypes as C
import os
import struct

import numpy as np
import pytest

import oracle_lib as O


def test_library_exports_every_declared_symbol(pkg):
    L = pkg.lib()
    names = pkg.declared_symbols()
    assert len(names) >= 60
    for n in names:
        assert hasattr(L, n), f"libpcnn.so does not export {n} declared in include/pcnn.h"
    assert L.pcnn_version() == 200


def test_sass_is_sm100a_only(pkg):
    import subprocess
    out = subprocess.run(["cuobjdump", "-lelf", pkg.LIB_PATH], capture_output=True, text=True).stdout
    archs = {tok for line in out.splitlines() for tok in line.replace(".", " ").split() if tok.startswith("sm_")}
    assert archs == {"sm_100a"}, archs


def test_init_params_reference_replays_glibc_rand(pkg, golden):
    p = pkg.init_params_reference()
    assert np.array_equal(p.view(np.uint32), golden["params_init"].view(np.uint32))   # the reference's constructor output
    assert np.array_equal(p.view(np.uint32), O.init_params().view(np.uint32))          # the real rand() after srand(1)


def test_create_without_gpu_fails_loudly(pkg):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        pytest.skip("a GPU is present")
    with pytest.raises(pkg.PcnnError) as ei:
        pkg.Engine(0)
    assert ei.value.code == -6 and "no CPU fallback" in str(ei.value)


def test_null_and_bad_arguments_are_rejected_without_a_context(pkg):
    L = pkg.lib()
    assert L.pcnn_sync(None) == -1
    assert L.pcnn_fp_c1(None, None, None, None, None, 1) == -1
    assert L.pcnn_train_step(None, 0, 1) == -1
    assert L.pcnn_init_params_reference(None) == -1
    assert b"NULL" in L.pcnn_last_error_string()
    assert L.pcnn_destroy(None) == 0


def _write_idx(tmp, images, labels, img_magic=2051, lab_magic=2049, lab_count=None, dims=(28, 28)):
    ip, lp = os.path.join(tmp, "img.idx"), os.path.join(tmp, "lab.idx")
    with open(ip, "wb") as f:
        f.write(struct.pack(">IIII", img_magic, len(images), dims[0], dims[1]))
        f.write(images.tobytes())
    with open(lp, "wb") as f:
        f.write(struct.pack(">II", lab_magic, len(labels) if lab_count is None else lab_count))
        f.write(labels.tobytes())
    return ip, lp


def test_mnist_loader_return_codes_follow_mnist_h(pkg, golden, tmp_path):
    tmp = str(tmp_path)
    imgs, labs = golden["train_u8"][:32], golden["train_labels"][:32]
    ip, lp = _write_idx(tmp, imgs, labs)
    rc, a, b = pkg.mnist_load_u8(ip, lp)
    assert rc == 0 and np.array_equal(a, imgs) and np.array_equal(b, labs)
    assert pkg.mnist_load_u8(os.path.join(tmp, "nope"), lp)[0] == -1            # mnist.h:95-98
    assert pkg.mnist_load_u8(*_write_idx(tmp, imgs, labs, img_magic=1234))[0] == -2   # mnist.h:100-104
    assert pkg.mnist_load_u8(*_write_idx(tmp, imgs, labs, lab_magic=1234))[0] == -3   # mnist.h:106-110
    assert pkg.mnist_load_u8(*_write_idx(tmp, imgs, labs, lab_count=31))[0] == -4     # mnist.h:118-121
    assert pkg.mnist_load_u8(*_write_idx(tmp, imgs, labs, dims=(28, 27)))[0] == -2    # mnist.h:128-131


def test_mnist_loader_reads_the_real_idx_files(pkg, golden, tmp_path):
    """IDX files of the MNIST test split's size and header (10,000 images of 28 x 28), filled with the 256 stored real test
    samples repeated in order."""
    te, tel = np.resize(golden["test_u8"], (10000, 784)), np.resize(golden["test_labels"], 10000)
    O.write_idx(str(tmp_path), te, tel, "t10k")
    rc, a, b = pkg.mnist_load_u8(str(tmp_path / "t10k-images.idx3-ubyte"), str(tmp_path / "t10k-labels.idx1-ubyte"))
    assert rc == 0 and a.shape == (10000, 784)
    assert np.array_equal(a, te) and np.array_equal(b, tel)


def test_sharding_covers_the_global_batch_exactly(pkg):
    from parallel_cnn_b200 import sharding as S
    n = 60000
    for B, world in [(1024, 8), (256, 2), (1000, 4), (1, 1), (7, 3)]:
        cursor, seen, steps = 0, 0, 0
        while True:
            ranges = [S.shard(cursor, B, r, world, n) for r in range(world)]
            got = sum(c for _, c in ranges)
            assert got == S.effective_global_batch(cursor, B, world, n)
            # contiguous, non-overlapping, in rank order
            pos = cursor
            for base, cnt in ranges:
                if cnt:
                    assert base == pos
                    pos += cnt
            seen += got
            steps += 1
            cursor = S.next_cursor(cursor, B, world, n)
            if cursor == 0:
                break
        assert seen == n and steps == S.steps_per_epoch(n, B, world)


# --------------------------------------------------------------------------- world_size-2 gloo test of the N > 1 path
def _dp_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import pcnn_loader
    pcnn_loader.load()
    from parallel_cnn_b200 import sharding as S
    d = np.load(os.path.join(O.GOLDEN, "mnist_subset.npz"))
    B, n = 16, 80                                   # 80 samples, global batch 32 -> 3 steps, the last one ragged (16 + 0)
    p = O.init_params()
    cursor = 0
    for _ in range(S.steps_per_epoch(n, B, world)):
        base, cnt = S.shard(cursor, B, rank, world, n)
        if cnt:
            g, es = O.batch_grad(p, O.u8_to_f32(d["train_u8"][base:base + cnt]), d["train_labels"][base:base + cnt])
        else:
            g, es = np.zeros(O.NPARAM), 0.0
        packed = torch.from_numpy(np.concatenate([g, [es]]))
        dist.all_reduce(packed)                      # the single exchange of the step
        lr = np.float32(0.1) / np.float32(S.effective_global_batch(cursor, B, world, n))
        p = O.apply_update(p, packed.numpy()[:O.NPARAM].astype(np.float32), lr)
        cursor = S.next_cursor(cursor, B, world, n)
    q.put((rank, p))
    dist.destroy_process_group()


def test_data_parallel_two_ranks_equal_single_process_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, q)) for r in range(2)]
    for pr in procs:
        pr.start()
    res = dict(q.get(timeout=120) for _ in range(2))
    for pr in procs:
        pr.join(timeout=60)
        assert pr.exitcode == 0
    # replicas identical
    assert np.array_equal(res[0].view(np.uint32), res[1].view(np.uint32))
    # and equal to one process doing the global batches
    d = np.load(os.path.join(O.GOLDEN, "mnist_subset.npz"))
    p = O.init_params()
    for lo in (0, 32, 64):
        hi = min(80, lo + 32)
        g, _ = O.batch_grad(p, O.u8_to_f32(d["train_u8"][lo:hi]), d["train_labels"][lo:hi])
        p = O.apply_update(p, g.astype(np.float32), np.float32(0.1) / np.float32(hi - lo))
    np.testing.assert_allclose(res[0], p, rtol=1e-6, atol=1e-7)


def test_conv_backward_tile_planning_is_host_logic(pkg):
    """pcnn_conv_bwd_plan_info needs no GPU: the tile shapes DESIGN.md 3.7 quotes for BASELINE config 5, and the shapes that must
    are refused (the FMA-pipe reference kernels run only after pcnn_conv_bwd_select)."""
    import ctypes as C

    def info(*shape):
        out = (C.c_int * 9)()
        assert pkg.lib().pcnn_conv_bwd_plan_info(*shape, out) == 0
        return list(out)

    cfg5 = info(128, 224, 224, 3, 64, 3, 3)
    assert cfg5[:4] == [1, 3, 112, 3]            # weight gradient: 3 dy rows x 112 pixels per tile (222 = 74 x 3, 2 x 112 >= 222), 3 stages
    assert cfg5[4:8] == [1, 2, 28, 4]            # input gradient: 2 strips of 112 columns, 28 outputs per lane quarter, 4 slot groups
    assert cfg5[8] >= 8
    k128 = info(4, 64, 64, 3, 128, 3, 3)
    assert k128[0] == 1 and k128[1] <= 2 and k128[4] == 1          # N = RB * 128 <= 256
    lenet = info(4, 28, 28, 1, 6, 5, 5)          # LeNet c1: 6 filters are zero-padded to 64 and run on the tensor-core kernels
    assert lenet[0] == 1 and lenet[4] == 1        # (given a row pitch that is a multiple of 8 elements)
    assert info(1, 32, 32, 3, 320, 3, 3)[0] == 0 and info(1, 32, 32, 3, 320, 3, 3)[4] == 0   # more than 256 filters: refused
    assert info(1, 32, 32, 3, 64, 5, 5)[0] == 0 and info(1, 32, 32, 3, 64, 5, 5)[4] == 1    # 5x5x3: 75 Hankel rows > 64


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the driver's reference arm) runs on host cores only and prints ONE JSON line with the keys the
    contract names; under torchrun only rank 0 prints."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RANK="0", WORLD_SIZE="1")
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--gpus", "1"],
                       capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "MNIST training images/sec" and d["unit"] == "images/s"
    assert d["higher_is_better"] is True and d["value"] > 100.0 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    r1 = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--gpus", "2"],
                        capture_output=True, text=True, timeout=120, env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert r1.returncode == 0 and r1.stdout.strip() == ""
