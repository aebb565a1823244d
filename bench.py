#!/usr/bin/env python
"""bench.py -- MNIST training images/s of the fused LeNet step on N B200s (BASELINE.json metric, config[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" is one pass of the hot path (forward + backward + packed-gradient reduction [+ all-reduce] + SGD update,
Main.cpp:157-171 batched) over one batch of B = 256 synthetic MNIST-shaped images per GPU.  Rank 0 prints ONE JSON line:

  value     whole-job images/s, inputs resident in HBM, K steps timed with CUDA events on the launching stream,
            bracketed by barrier + synchronize, max over ranks
  e2e       the same metric through the public host-buffer API (Engine.learn_host = pcnn_learn_host): every step's
            u8 images + labels are copied from PINNED host memory inside the timed region (chunked, double-buffered
            copy stream) and every step's error sum is read back to the host
  roofline  fused gradient kernel alone: algorithmic flops / bytes per launch over its average duration (CUDA events,
            pcnn_time_fused_kernel), against the fp32 FMA rate measured live on this GPU and the measured HBM peak
            of MEASURED_PEAKS.json.  The fused LeNet step is fp32-FMA bound (AI = 122 flop/B, SURVEY.md 8d); both
            fractions are reported, `bound` names the larger one
  cpu_baseline  the unmodified reference (oracle/_ref, else the oracle port) timed on one host core on a bounded sample
  clocks    nvidia-smi SM clock / throttle reasons sampled while the GPU phases run

--impl reference times the reference's own CPU implementation (all host cores, independent replicas) for the same
metric; rank 0 only under torchrun.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOPS_PER_IMAGE = 383948            # SURVEY.md 8d: fused train step, 191,974 MAC
BYTES_PER_IMAGE_U8 = 788            # 784 B image + 4 B label (SURVEY.md 8d); fp32 input would be 3,140
PARAM_BYTES = 2344 * 4              # packed parameters read once per CTA-wave; counted once per launch
DATASET_IMAGES = 262144             # 205 MB of u8 images > 126 MB L2: every step reads its batch from HBM


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for ts, r in self.rows if t0 <= ts <= t1] or [r for _, r in self.rows]
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_traffic(kernel, batch, steps):
    """DRAM bytes of one launch from profiles/traffic.json ({kernel: {batch: bytes_per_step}}), or None."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        return float(d[kernel][str(batch)]["dram_bytes_per_step"]) * steps
    except Exception:
        return None


def dump_outputs(directory, eng):
    """What the timed steps leave for a caller of Engine.train_steps, read back after the last one: the packed parameters
    they updated, the packed gradient of the last step and the running sum of per-sample error norms.  The inputs depend
    only on the arguments, so two builds of the project can be compared file for file."""
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "params.npy"), eng.get_params())
    np.save(os.path.join(directory, "grads.npy"), eng.get_grads())
    np.save(os.path.join(directory, "err_sum.npy"), np.array([eng.err_sum()], np.float64))


def synthetic(n, seed):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 256, (n, 784), dtype=np.uint8), rng.integers(0, 10, n, dtype=np.uint8)


def load_training_set():
    """Seeded synthetic MNIST-shaped bytes, the same on every run whatever else lies in the tree, so that runs of two builds
    see identical inputs; the device-resident set (205 MB) is larger than the 126 MB L2, so every step reads its batch
    from HBM.  Returns (images u8 [n,784], labels u8 [n], description)."""
    imgs, labs = synthetic(DATASET_IMAGES, 7)
    return imgs, labs, "synthetic"


def host_cores():
    """CPUs this process may actually use: scheduler affinity, capped by the cgroup CPU quota (a 1-GPU lease can report
    128 CPUs and grant a dozen).  Returns (count, sorted affinity list, description)."""
    aff = sorted(os.sched_getaffinity(0))
    n, why = len(aff), f"affinity {len(aff)} of {os.cpu_count()}"
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                quota, period = txt[0], float(txt[1])
            else:
                quota, period = txt[0], float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota not in ("max", "-1"):
                q = max(1, int(float(quota) / period))
                if q < n:
                    n, why = q, why + f", cgroup quota {float(quota) / period:.1f} CPUs"
            break
        except Exception:
            continue
    return n, aff, why


# ----------------------------------------------------------------------------------------------- reference arm
def _ref_worker(args):
    """One host core (pinned): the unmodified reference (or the oracle port) trains on `n` samples per step."""
    wid, cpu, n, steps, warmup, native = args
    if cpu is not None:
        try:
            os.sched_setaffinity(0, {cpu})
        except Exception:
            pass
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    imgs, labs, _ = load_training_set()
    lo = (wid * n) % max(1, imgs.shape[0] - n)
    imgs, labs = np.ascontiguousarray(imgs[lo:lo + n]), np.ascontiguousarray(labs[lo:lo + n])
    ref = O.reference(native=native)
    secs = np.zeros(1, np.float64)
    if ref is not None:
        run = lambda: ref.ref_learn_loop_u8(O.u8p(imgs.reshape(-1)), O.u8p(labs), n, O.dp(secs))
    else:
        p = O.init_params()
        run = lambda: O.oracle().orc_learn(O.fp(p), O.u8p(imgs.reshape(-1)), O.u8p(labs), n)
    for _ in range(warmup):
        run()
    t0 = time.perf_counter()
    for _ in range(steps):
        run()
    return time.perf_counter() - t0


def cpu_reference_throughput(cores, cpu_list, n_per_step, steps, warmup, native=False):
    import multiprocessing as mp
    jobs = [(w, cpu_list[w % len(cpu_list)] if cpu_list else None, n_per_step, steps, warmup, native) for w in range(cores)]
    with mp.get_context("fork").Pool(cores) as pool:
        times = pool.map(_ref_worker, jobs)
    return cores * steps * n_per_step / max(times), max(times)


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    kind = "reference" if O.reference() is not None else "port"
    cores, aff, why = host_cores()
    _, _, data = load_training_set()
    # bounded sample: ~60 s of CPU work in total at ~4.4 k img/s/core (BASELINE.md section 2)
    n_per_step = int(max(8, min(4096, 60.0 * 4400 / max(1, a.steps + a.warmup))))
    value, secs = cpu_reference_throughput(cores, aff, n_per_step, a.steps, a.warmup)
    line = {
        "impl": "reference", "metric": "MNIST training images/sec", "value": value, "unit": "images/s",
        "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * secs / a.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": data,
        "config": {"workload": "lenet_mnist_train_fp32_fused_step (BASELINE.json configs[1])", "reference_batch": 1,
                   "note": "the reference's own CPU implementation of the same workload: Sequential/Main.cpp learn() loop; "
                           "batch-1 per-sample SGD is the only mode the reference has"},
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": cores, "kind": kind, "cores_how": why,
                         "sample": f"{cores} independent single-thread replicas (one per granted CPU, pinned with "
                                   f"sched_setaffinity) x {n_per_step} samples per step, g++ -O2"},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- our arm
def conv_roofline(eng, pkg, stream, hbm_peak, peak_src, n_img=128, iters=10):
    """BASELINE.json's second metric: HBM GB/s of the conv forward + weight gradient + input gradient against the roofline, on
    configs[4] (synthetic 224x224x3 -> 64 filters 3x3, bf16 NHWC, valid padding; SURVEY.md 8d: 6,609,408 algorithmic bytes per
    image per pass).  Every pass streams 846 MB (> 126 MB L2); CUDA events on the engine's stream, 3 warm-up launches."""
    import torch
    N, H, W, C, K, R, S = n_img, 224, 224, 3, 64, 3, 3
    P, Q = H - R + 1, W - S + 1
    g = torch.Generator(device="cuda").manual_seed(1234)
    x = (torch.rand((N, H, W, C), device="cuda", generator=g)).to(torch.bfloat16)                 # x ~ U[0,1)
    f = torch.rand((K, R, S, C), device="cuda", generator=g) - 0.5                                 # w ~ U[-0.5,0.5)
    yb = torch.empty((N, P, Q, K), dtype=torch.bfloat16, device="cuda")
    dw = torch.empty((K, R, S, C), dtype=torch.float32, device="cuda")
    dx = torch.empty((N, H, W, C), dtype=torch.bfloat16, device="cuda")
    plan = pkg.ConvPlan(eng, N, H, W, C, K, R, S, f.cpu().numpy(), None, act=0, row_pitch=W * C)
    alg = N * (H * W * C + P * Q * K) * 2
    out = {}

    def timed(fn):
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

    ms_f = timed(lambda: plan.fwd(x, yb))
    dy = yb                                                                                        # the forward output doubles as dy
    ms_w = timed(lambda: eng.conv_wgrad(x, dy, dw, N, H, W, C, K, R, S))
    ms_d = timed(lambda: eng.conv_dgrad(dy, f, dx, N, H, W, C, K, R, S))
    plan.close()
    for name, ms in (("fwd", ms_f), ("wgrad", ms_w), ("dgrad", ms_d)):
        gb = alg / (ms * 1e-3) / 1e9
        out[name] = {"ms": ms, "GBps": gb, "frac": gb / hbm_peak}
    tot = ms_f + ms_w + ms_d
    gb = 3 * alg / (tot * 1e-3) / 1e9
    return {"workload": "conv 224x224x3 -> 64x3x3, bf16 NHWC, tcgen05 kernels (BASELINE.json configs[4])", "images": N,
            "algorithmic_bytes_per_pass": alg, "passes": out, "fwd_bwd": {"ms": tot, "GBps": gb, "frac": gb / hbm_peak},
            "peak": hbm_peak, "unit": "GB/s", "peak_source": peak_src, "l2": "846 MB per pass, larger than L2"}


def reference_cuda_baseline(samples=20000):
    """The reference's own GPU path (CUDA/main.cu + layer.cu, unmodified, built for sm_100a by oracle/Makefile) timed on
    this B200 with a device synchronise around learn() -- batch 1, ~38 driver calls per image (SURVEY.md 2.2).  Baseline
    only: it is numerically wrong in two kernels and is never used as a checker."""
    exe = os.path.join(ROOT, "oracle", "_ref", "cuda_ref_bench")
    if not os.path.exists(exe):
        return None
    try:
        r = subprocess.run([exe, str(samples)], cwd=os.path.join(ROOT, "oracle", "_ref"), capture_output=True, text=True, timeout=300)
        for ln in r.stdout.splitlines():
            if ln.startswith("REF_CUDA"):
                kv = dict(x.split("=") for x in ln.split()[1:])
                return {"value": float(kv["images_per_s"]), "unit": "images/s", "samples": int(kv["samples"]),
                        "seconds": float(kv["seconds"]), "kind": "reference CUDA/ (unmodified, sm_100a, batch 1, device-synchronised wall clock)"}
        return {"unavailable": (r.stderr or r.stdout)[-200:]}
    except Exception as exc:
        return {"unavailable": str(exc)[:200]}


def run_ours(a):
    import torch
    import pcnn_loader
    pkg = pcnn_loader.load()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus:
        raise SystemExit(f"--gpus {a.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {a.gpus}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    # a non-default torch stream: torch.cuda.Event then times exactly the stream the kernels are launched on
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    eng = pkg.Engine(local, stream.cuda_stream)
    B, K, W = a.batch, a.steps, max(a.warmup, 3)

    # the training set, identical on every rank: ranks read disjoint windows of every global batch
    imgs, labs, data_desc = load_training_set()
    n_data = imgs.shape[0]
    eng.dataset_upload(pkg.TRAIN_SET, imgs, labs)
    if world > 1:
        if a.mode == "graph":        # per-step kernels in CUDA graphs + one ncclAllReduce of the packed gradient per step
            uid = [pkg.Engine.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            eng.comm_init_rank(uid[0], rank, world)
        else:                        # persistent kernel, gradient chunks exchanged in-kernel over NVLink peer memory
            handles = [None] * world
            dist.all_gather_object(handles, eng.p2p_export())
            ok = 1
            try:
                eng.p2p_attach(handles, rank, world)
            except pkg.PcnnError as exc:             # e.g. CUDA IPC not permitted in this container
                ok = 0
                if rank == 0:
                    print(f"bench.py: peer attach failed ({exc}); falling back to graph + NCCL", file=sys.stderr)
            flag = torch.tensor([ok], device="cuda")
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if int(flag.item()) == 0:                # all ranks take the same path
                if ok:
                    eng.p2p_detach()
                uid = [pkg.Engine.comm_unique_id() if rank == 0 else None]
                dist.broadcast_object_list(uid, src=0)
                eng.comm_init_rank(uid[0], rank, world)
                a.mode = "graph"
    eng.set_step_mode({"auto": pkg.MODE_AUTO, "graph": pkg.MODE_GRAPH, "persistent": pkg.MODE_PERSISTENT}[a.mode])
    if a.persist_tune:
        eng.persist_tune(a.persist_tune)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def aligned_start():
        """All ranks leave at the same instant of the node's monotonic clock (single node: one clock): a collective barrier
        alone releases the ranks tens of microseconds apart, which a short timed region would count as step time."""
        if world == 1:
            return
        tgt = torch.tensor([time.monotonic() + 0.003], dtype=torch.float64, device="cuda")
        dist.broadcast(tgt, src=0)
        t_go = float(tgt.item())
        while time.monotonic() < t_go:
            pass

    def timed_steps(batch, k, w):
        """w warm-up + k timed cursor-driven steps of `batch` images per GPU; returns ms (max over ranks)."""
        eng.train_steps_prepare(batch, k)
        eng.train_steps(0, batch, w)
        barrier()
        aligned_start()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record(stream)
        eng.train_steps(-1, batch, k)
        a1.record(stream)
        barrier()
        t_ms = a0.elapsed_time(a1)
        if world > 1:
            tt = torch.tensor([t_ms], device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t_ms = float(tt.item())
        return t_ms

    # ---- multi-GPU parity, where the driver sees it (SURVEY.md 8a x4): 4 data-parallel steps of 1024 images per GPU
    # against the same global batch on ONE GPU (a second, unattached engine on rank 0); replicas must be bit-identical
    parity = None
    if world > 1:
        PB, PK = 1024, 4
        p0 = pkg.init_params_reference()
        eng.set_params(p0)
        barrier()
        eng.train_steps(0, PB, PK)
        eng.sync()
        p_dp = eng.get_params()
        bits = torch.from_numpy(p_dp.view(np.int32).copy()).cuda()
        lo, hi = bits.clone(), bits.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        identical = bool(torch.equal(lo, hi))
        rel = 0.0
        if rank == 0:
            n_sub = PB * world * PK
            with pkg.Engine(local) as solo:
                solo.dataset_upload(pkg.TRAIN_SET, imgs[:n_sub], labs[:n_sub])
                solo.set_params(p0)
                solo.train_steps(0, PB * world, PK)
                solo.sync()
                p_1 = solo.get_params()
            rel = float(np.linalg.norm(p_dp.astype(np.float64) - p_1) / np.linalg.norm(p_1.astype(np.float64)))
        parity = {"rel_l2_params": rel, "replicas_bit_identical": identical, "global_batch": PB * world, "steps": PK,
                  "bound": 1e-6, "against": "one GPU training the same global batch (second engine on rank 0)"}
        ok = torch.tensor([1 if (identical and rel <= 1e-6) else 0], device="cuda")
        dist.broadcast(ok, src=0)
        if int(ok.item()) == 0:
            if rank == 0:
                print(json.dumps({"error": "multi-GPU parity failed", "parity": parity}), flush=True)
            raise SystemExit(3)
        eng.set_params(p0)
        barrier()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()

    # the fp32 FMA rate of this GPU under its current clocks (the roofline's denominator), measured BEFORE the timed regions:
    # ~15 ms of dense FFMA also takes the GPU out of its idle clock state, which a 20-step timed region (0.2 ms) would
    # otherwise still be ramping out of
    fp32_peak = eng.measure_fp32_peak()

    # ---- value: device-resident inputs
    eng.train_steps_prepare(B, K)            # instantiate the step graphs the timed call replays (host work, untimed)
    eng.train_steps(0, B, W)                 # W untimed warm-up steps
    barrier()
    aligned_start()
    l0 = eng.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.time()
    e0.record(stream)
    eng.train_steps(-1, B, K)                # exactly K steps, continuing at the device-side sample cursor
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    launches = eng.launch_count() - l0
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = K * B * world / (ms * 1e-3)
    if a.dump_outputs and rank == 0:         # replicas are identical after every step
        dump_outputs(a.dump_outputs, eng)

    # ---- e2e: pinned host buffers through the public host API (single-GPU entry point; per-rank shard when N > 1)
    K2 = min(K, 8192)                        # bounds the pinned host buffer (8192 steps x 256 x 784 B = 1.6 GB)
    n_e2e = K2 * B
    hi = torch.empty((n_e2e, 784), dtype=torch.uint8, pin_memory=True)
    hl = torch.empty((n_e2e,), dtype=torch.uint8, pin_memory=True)
    sel = (np.arange(n_e2e) + rank * n_e2e) % n_data                # every rank streams its own shard
    hi.numpy()[:] = imgs[sel]
    hl.numpy()[:] = labs[sel]
    eng.learn_host(hi.numpy(), hl.numpy(), B=B, epochs=1)            # warm-up pass (graphs, staging buffers)
    barrier()
    aligned_start()
    t0 = time.perf_counter()
    eng.learn_host(hi.numpy(), hl.numpy(), B=B, epochs=1)            # returns when the last step's result is on the host
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    assert eng.step_errs().shape[0] == K2
    if world > 1:
        t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_val = n_e2e * world / e2e_s
    barrier()
    # the host->device link as this box gives it (pinned memory, one copy, CUDA events): the ceiling of ANY end-to-end number,
    # because every step needs B x 785 bytes across it.  Measured for 64 MB and for exactly the bytes the e2e call moved.
    link = None
    if rank == 0:
        def h2d_gbps(nbytes):
            src = torch.empty((nbytes,), dtype=torch.uint8, pin_memory=True)
            dst = torch.empty((nbytes,), dtype=torch.uint8, device="cuda")
            best = 0.0
            for _ in range(4):
                c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                c0.record(stream)
                dst.copy_(src, non_blocking=True)
                c1.record(stream)
                torch.cuda.synchronize()
                best = max(best, nbytes / (c0.elapsed_time(c1) * 1e-3) / 1e9)
            return best
        big, same = h2d_gbps(64 << 20), h2d_gbps(n_e2e * 785)
        bound = same * 1e9 / 785.0 * world
        link = {"h2d_GBps_64MB": big, "h2d_GBps_same_bytes_one_copy": same, "link_bound_images_per_s": bound,
                "e2e_frac_of_link_bound": e2e_val / bound,
                "note": "one cudaMemcpyAsync of the e2e call's input bytes, nothing else: the rate at which this box's link can "
                        "deliver pixels; every step needs B x 785 of them"}
    barrier()

    # ---- BASELINE.json configs[3]: 1024 images per GPU (weak) and a fixed global batch of 8192 (strong)
    b1024 = None
    if not a.no_batch1024:
        K4 = max(50, min(K, 1000))
        ms_w = timed_steps(1024, K4, 20)
        bs = 8192 // world
        ms_s = ms_w if bs == 1024 else timed_steps(bs, K4, 20)
        b1024 = {"weak_1024_per_gpu": {"value": K4 * 1024 * world / (ms_w * 1e-3), "ms_per_step": ms_w / K4, "global_batch": 1024 * world},
                 "strong_global_8192": {"value": K4 * 8192 / (ms_s * 1e-3), "ms_per_step": ms_s / K4, "batch_per_gpu": bs},
                 "steps": K4, "unit": "images/s",
                 "parity_note": "batches beyond the oracle's reach are covered by additivity / determinism tests (tests/test_fused_gpu.py)"}

    # ---- phase trace of the persistent kernel at this N (CTA 0 of every rank; rank 0's is printed): where a step's time goes
    phases = None
    if a.mode != "graph" and not a.no_phase_trace:
        eng.train_steps(0, B, 50)
        barrier()
        eng.persist_trace_arm()
        eng.train_steps(-1, B, 256)
        eng.sync()
        tr = eng.persist_trace_read(256)[8:]
        dd = np.diff(tr, axis=1).astype(np.float64) / 1e3
        stepus = np.diff(tr[:, 0]).astype(np.float64) / 1e3
        names = ["param_fetch", "images", "epilogue+cluster_reduce", "owner_gather", "exchange+update+publish"]
        phases = {"step_us_median": float(np.median(stepus)), "unit": "us", "view": "CTA 0 of rank 0, %globaltimer (0.26 us resolution)"}
        phases.update({n: float(np.median(dd[:, i])) for i, n in enumerate(names)})
        phases.update(eng.persist_info())
        barrier()

    # ---- roofline of the dominant kernel + live fp32 peak
    line = None
    if rank == 0:
        k_ms = eng.time_fused_kernel(B, max(200, min(K, 5000)))
        t_gpu_end = time.time()
        clocks = sampler.stop(t_wall0, t_gpu_end)
        hbm_peak, peak_src = peaks()
        # dominant kernel of the timed region: in persistent mode ONE launch of k_train_persist runs all K steps (its
        # duration is the CUDA-event time of the region); in graph mode it is k_fused, timed alone right above
        persistent = a.mode != "graph"
        if persistent:
            kernel, launch_ms, launch_steps = "k_train_persist<u8> (K steps per launch)", ms, K
        else:
            kernel, launch_ms, launch_steps = "k_fused<u8,train>", k_ms, 1
        flops = launch_steps * B * FLOPS_PER_IMAGE                       # per GPU
        bytes_alg = launch_steps * (B * BYTES_PER_IMAGE_U8 + 2 * PARAM_BYTES)
        tf = flops / (launch_ms * 1e-3) / 1e12
        gbs = bytes_alg / (launch_ms * 1e-3) / 1e9
        frac_f, frac_h = tf / fp32_peak, gbs / hbm_peak
        roof = {"bound": "fp32_fma" if frac_f >= frac_h else "hbm",
                "achieved": tf if frac_f >= frac_h else gbs, "peak": fp32_peak if frac_f >= frac_h else hbm_peak,
                "unit": "TFLOP/s" if frac_f >= frac_h else "GB/s", "frac": max(frac_f, frac_h),
                # dram__bytes_read.sum + dram__bytes_write.sum of this kernel per step, read from the summary that
                # scripts/ncu_traffic.py wrote from the round's `ncu --set full` capture (null when no capture matches)
                "traffic": measured_traffic("k_train_persist" if persistent else "k_fused", B, launch_steps),
                "kernel": kernel, "kernel_ms": launch_ms,
                "fp32": {"achieved": tf, "peak": fp32_peak, "unit": "TFLOP/s", "frac": frac_f,
                         "peak_source": "measured live (pcnn_measure_fp32_peak FFMA micro-benchmark)"},
                "hbm": {"achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": frac_h, "peak_source": peak_src},
                "algorithmic_per_launch": {"flops": flops, "bytes": bytes_alg},
                "fused_kernel_alone": {"kernel": "k_fused<u8,train>", "ms": k_ms,
                                       "tflops": B * FLOPS_PER_IMAGE / (k_ms * 1e-3) / 1e12}}
        # ---- CPU baseline beside it (N = 1 only): the unmodified reference on ONE host core
        cpu = None
        ref_gpu = None
        if world == 1 and not a.no_cpu_baseline:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import oracle_lib as O
            kind = "reference" if O.reference() is not None else "port"
            n_cpu = 40000
            ncores, aff, why = host_cores()
            v, secs = cpu_reference_throughput(1, aff[:1], n_cpu, 1, 0)
            cpu = {"value": v, "unit": "images/s", "cores": 1, "kind": kind,
                   "sample": f"{n_cpu} MNIST samples, Sequential/Main.cpp learn() loop (batch 1), g++ -O2, {secs:.1f} s",
                   "host_cores_granted": ncores, "host_cores_how": why}
            if O.reference(native=True) is not None:      # BASELINE.md 3.2: best single-core build of the same sources
                v3, s3 = cpu_reference_throughput(1, aff[:1], n_cpu, 1, 0, native=True)
                cpu["native_O3"] = {"value": v3, "flags": "-O3 -march=x86-64-v3 (FMA contraction: timing only)", "seconds": s3}
            ref_gpu = reference_cuda_baseline()
        conv = None
        if world == 1 and not a.no_conv:
            conv = conv_roofline(eng, pkg, stream, hbm_peak, peak_src)
        line = {
            "metric": "MNIST training images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "fp32", "data": data_desc,
            "config": {"workload": "lenet_mnist_train_fp32_fused_step (BASELINE.json configs[1])", "batch_per_gpu": B,
                       "global_batch": B * world, "pixel_type": "u8", "parallelism": f"dp{world}",
                       "step_mode": ("graph+nccl" if world > 1 else "graph") if a.mode == "graph" else
                                    ("persistent+nvlink_p2p" if world > 1 else "persistent"),
                       "l2": f"inputs larger than L2: steps walk a {n_data}-image ({n_data * 784 / 1e6:.0f} MB) device-resident set",
                       "update": "w += (dt / global_batch) * sum_b g_b, dt = 0.1 (equals the reference at batch 1)"},
            "e2e": {"value": e2e_val, "unit": "images/s", "h2d_bytes_per_step": B * 785 * world,
                    "d2h_bytes_per_step": 4 * world, "steps": K2, "api": "Engine.learn_host (pcnn_learn_host), pinned host u8: the training kernel pulls each step's images across PCIe itself (cp.async.bulk from the pinned buffer); labels by one H2D copy; per-step results written to mapped host memory",
                    "link": link},
            "gpu_launches": launches, "roofline": roof, "cpu_baseline": cpu, "ref_gpu_baseline": ref_gpu, "clocks": clocks,
            "parity": parity, "batch1024": b1024, "phase_trace": phases, "conv": conv,
        }
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--batch", type=int, default=256, help="images per GPU per step (BASELINE.json configs[1]: 256)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-conv", action="store_true", help="skip the conv fwd+bwd roofline block (N = 1 only)")
    ap.add_argument("--persist-tune", type=int, default=0, help="pcnn_persist_tune knob (profiling runs: 2 = clusters without the cooperative attribute)")
    ap.add_argument("--no-phase-trace", action="store_true", help="skip the per-phase trace of the persistent kernel")
    ap.add_argument("--no-batch1024", action="store_true", help="skip the 1024-per-GPU / global-8192 block")
    ap.add_argument("--mode", default="auto", choices=["auto", "graph", "persistent"],
                    help="auto/persistent: one cooperative kernel runs all K steps (N > 1: in-kernel NVLink exchange); "
                         "graph: per-step kernels replayed from CUDA graphs (N > 1: ncclAllReduce per step)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what they computed as DIR/params.npy, grads.npy, err_sum.npy")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if a.impl == "reference":
        run_reference_arm(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
