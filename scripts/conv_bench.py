#!/usr/bin/env python
"""scripts/conv_bench.py -- throughput of the bf16 tcgen05 convolution forward (BASELINE.json configs 3 and 5) against the
HBM roofline.  Algorithmic bytes per image are SURVEY.md 8d's: each operand crosses HBM once (input read + output written,
bf16): LeNet c1 8,480 B, 224x224x3 -> 64 x 3x3: 6,609,408 B.  CUDA-event timing over back-to-back launches after warm-up;
the working set of every measured point except the smallest batches exceeds the 126 MB L2."""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pcnn_loader  # noqa: E402

pkg = pcnn_loader.load()
torch.cuda.set_device(0)
stream = torch.cuda.Stream()
torch.cuda.set_stream(stream)
eng = pkg.Engine(0, stream.cuda_stream)
HBM = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"] if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0
rng = np.random.default_rng(1234)
only = sys.argv[1] if len(sys.argv) > 1 else "all"


def run(name, N, H, W, C, K, R, S, act, iters, image_rows=0, bias=True):
    pitch = (W * C + 7) // 8 * 8
    P, Q = H - R + 1, W - S + 1
    f = rng.uniform(-0.5, 0.5, (K, R, S, C)).astype(np.float32)
    b = rng.uniform(-0.5, 0.5, K).astype(np.float32)
    plan = pkg.ConvPlan(eng, N, H, W, C, K, R, S, f, b if bias else None, act=act, row_pitch=pitch, image_rows=image_rows)
    x = torch.randint(0, 0x3F80, (N * (image_rows or H), pitch), dtype=torch.int16, device="cuda")   # positive bf16 bit patterns < 1.0
    y = torch.empty((N, P, Q, K), dtype=torch.int16, device="cuda")
    for _ in range(3):
        plan.fwd(x, y)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(iters):
        plan.fwd(x, y)
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    alg = N * (H * W * C + P * Q * K) * 2                       # bf16 in + out, once each
    flops = 2.0 * N * P * Q * K * R * S * C
    row = {"case": name, "N": N, "ms": ms, "img_per_s": N / (ms * 1e-3), "alg_GBps": alg / (ms * 1e-3) / 1e9,
           "hbm_frac": alg / (ms * 1e-3) / 1e9 / HBM, "useful_TFLOPs": flops / (ms * 1e-3) / 1e12,
           "working_set_MB": (N * H * pitch + N * P * Q * K) * 2 / 1e6}
    print(json.dumps(row), flush=True)
    plan.close()
    del x, y


def run_bwd(name, N, H, W, C, K, R, S, iters, stride=1, path="tc"):
    """wgrad and dgrad of the same layer: algorithmic bytes = dy read + x read (wgrad) / dy read + dx written (dgrad), bf16.
    stride: the window step (dy [N][(H-R)/stride+1][(W-S)/stride+1][K]); path "fma" selects the FMA-pipe reference kernels."""
    P, Q = (H - R) // stride + 1, (W - S) // stride + 1
    xb = torch.randint(0, 0x3F80, (N, H, W, C), dtype=torch.int16, device="cuda")
    dyb = torch.randint(0, 0x3F80, (N, P, Q, K), dtype=torch.int16, device="cuda")
    dyb ^= (torch.randint(0, 2, (N, P, Q, K), dtype=torch.int16, device="cuda") << 15)      # random signs
    f = torch.rand((K, R, S, C), dtype=torch.float32, device="cuda") - 0.5
    dw = torch.empty((K, R, S, C), dtype=torch.float32, device="cuda")
    dx = torch.empty((N, H, W, C), dtype=torch.int16, device="cuda")
    alg = N * (H * W * C + P * Q * K) * 2
    flops = 2.0 * N * P * Q * K * R * S * C
    eng.conv_bwd_select(reference=(path == "fma"))
    for what, fn in (("wgrad", lambda: eng.conv_wgrad(xb, dyb, dw, N, H, W, C, K, R, S, stride=stride)),
                     ("dgrad", lambda: eng.conv_dgrad(dyb, f, dx, N, H, W, C, K, R, S, stride=stride))):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        import time
        e0.record(stream)
        t0 = time.perf_counter()
        for _ in range(iters):
            fn()
        host_us = (time.perf_counter() - t0) / iters * 1e6           # host time to enqueue one call
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        print(json.dumps({"case": name + " " + what, "host_enqueue_us": host_us, "N": N, "ms": ms, "img_per_s": N / (ms * 1e-3), "alg_GBps": alg / (ms * 1e-3) / 1e9,
                          "hbm_frac": alg / (ms * 1e-3) / 1e9 / HBM, "useful_TFLOPs": flops / (ms * 1e-3) / 1e12,
                          "path": path, "stride": stride, "working_set_MB": alg / 1e6}), flush=True)
    eng.conv_bwd_select(reference=False)
    del xb, dyb, dx


if only in ("all", "bwd"):
    for N in (8, 32, 128):
        run_bwd("224x224x3->64x3x3 bf16 (config 5)", N, 224, 224, 3, 64, 3, 3, 10)
if only == "bwdpad":                                                   # filter counts padded to 64: 32 filters, and LeNet's own 6
    run_bwd("224x224x3->32x3x3 bf16 (padded to 64 filters)", 128, 224, 224, 3, 32, 3, 3, 10)
    run_bwd("224x224x3->16x3x3 bf16 (padded to 64 filters)", 128, 224, 224, 3, 16, 3, 3, 10)
if only == "bwdk128":                                                  # 128 filters: two 64-filter groups per dy row
    run_bwd("224x224x3->128x3x3 bf16", 64, 224, 224, 3, 128, 3, 3, 10)
if only == "bwds":                                                     # strided backward passes (config 5 at stride 2) next to stride 1
    import subprocess
    q = subprocess.run(["nvidia-smi", "--id=%d" % torch.cuda.current_device(), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print(json.dumps({"case": "device", "torch_name": torch.cuda.get_device_name(), "nvidia_smi_name_power_limit_max_sm_clock": q,
                      "hbm_peak_GBps_used_for_hbm_frac": HBM}), flush=True)
    for N in (32, 128):
        run_bwd("224x224x3->64x3x3/2 bf16 (config 5, stride 2)", N, 224, 224, 3, 64, 3, 3, 10, stride=2)
    run_bwd("224x224x3->64x3x3/2 bf16 (config 5, stride 2)", 8, 224, 224, 3, 64, 3, 3, 2, stride=2, path="fma")
    for N in (32, 128):
        run_bwd("224x224x3->64x3x3 bf16 (config 5)", N, 224, 224, 3, 64, 3, 3, 10)
    run_bwd("224x224x3->64x3x3 bf16 (config 5)", 8, 224, 224, 3, 64, 3, 3, 2, path="fma")
if only == "bwd128":                                                   # the profiler's target: few launches
    run_bwd("224x224x3->64x3x3 bf16 (config 5)", 128, 224, 224, 3, 64, 3, 3, 2)
if only in ("all", "lenet"):
    for N in (1024, 8192, 65536):
        run("lenet_c1_bf16_sigmoid (config 3 shape)", N, 28, 28, 1, 6, 5, 5, 1, 20)
    for N in (8192, 65536):
        run("lenet_c1_bf16_sigmoid, 32-row image pitch (TMA-store epilogue)", N, 28, 28, 1, 6, 5, 5, 1, 20, image_rows=32)
if only == "lenet1024":                                                # BASELINE configs[2]: LeNet c1 shape, batch 1024
    run("lenet_c1_bf16_sigmoid (config 3 shape)", 1024, 28, 28, 1, 6, 5, 5, 1, 2)
if only == "fwd128":                                                   # the profiler's target
    run("224x224x3->64x3x3 bf16 (config 5)", 128, 224, 224, 3, 64, 3, 3, 0, 2)
if only == "stprobe":                                                  # the store phase of the forward epilogue alone
    N, P, H, RE = 128, 222, 224, 222 * 64
    y = torch.empty((N, P, RE), dtype=torch.int16, device="cuda")
    for mode in (0, 2, 5, 6):
        for hot in (0, 1):
            g = eng.measure_tma_write(y, N, P, H, RE, mode, hot, 10)
            print(json.dumps({"case": "tma store probe", "mode": mode, "hot_l2_target": hot, "GBps": g, "us_per_launch": N * P * RE * 2 / g / 1e3}), flush=True)
if only == "fwdq":                                                     # one line: forward at N = 128 without bias
    run("224x224x3->64x3x3 bf16 (config 5), no bias", 128, 224, 224, 3, 64, 3, 3, 0, 20, bias=False)
if only == "fwdab":                                                    # forward at N = 128: with / without bias, with sigmoid
    run("224x224x3->64x3x3 bf16 (config 5), bias", 128, 224, 224, 3, 64, 3, 3, 0, 20)
    run("224x224x3->64x3x3 bf16 (config 5), no bias", 128, 224, 224, 3, 64, 3, 3, 0, 20, bias=False)
    run("224x224x3->64x3x3 bf16 (config 5), bias + sigmoid", 128, 224, 224, 3, 64, 3, 3, 1, 20)
    run("lenet_c1_bf16_sigmoid, 32-row image pitch (TMA-store epilogue)", 65536, 28, 28, 1, 6, 5, 5, 1, 20, image_rows=32)
    run("lenet_c1_bf16_sigmoid (config 3 shape)", 65536, 28, 28, 1, 6, 5, 5, 1, 20)
if only in ("all", "cfg5"):
    for N in (1, 8, 32, 128):
        run("224x224x3->64x3x3 bf16 (config 5)", N, 224, 224, 3, 64, 3, 3, 0, 10)
eng.close()
if only == "wprobe":                                                   # what a pure WRITE stream / pure READ stream / copy reach on this GPU
    # library fill / reduce / copy kernels as a yardstick for the store-dominated forward pass (807 MB written, 39 MB read):
    # MEASURED_PEAKS.json's HBM number is a COPY (half reads, half writes)
    nbytes = 807 << 20
    buf = torch.empty((nbytes // 4,), dtype=torch.int32, device="cuda")
    src = torch.ones((nbytes // 4,), dtype=torch.int32, device="cuda")
    def timeit(fn, iters=20):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(iters):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters
    ms_fill = timeit(lambda: buf.fill_(7))
    ms_memset = timeit(lambda: buf.zero_())
    ms_copy = timeit(lambda: buf.copy_(src))
    ms_read = timeit(lambda: src.sum())
    print(json.dumps({"case": "write/read/copy yardsticks (torch library kernels, 807 MiB)", "fill_GBps": nbytes / ms_fill / 1e6,
                      "memset_GBps": nbytes / ms_memset / 1e6, "copy_GBps_read_plus_write": 2 * nbytes / ms_copy / 1e6,
                      "reduce_read_GBps": nbytes / ms_read / 1e6, "hbm_peak_file": HBM}), flush=True)
