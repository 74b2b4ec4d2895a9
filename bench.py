#!/usr/bin/env python
"""bench.py -- roko hot-path throughput on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch 128] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A *step* is one pass of the hot path (front end -> 3 x (projection, recurrence) -> head+argmax) over
one batch of synthetic windows; the timed region is exactly K steps.  ``--dump-outputs DIR`` writes
the labels of the last timed step (what ``RNN.predict`` returns to its caller) as ``DIR/labels.npy``
(float32); the inputs are seeded, so two builds run with the same arguments can be compared output
for output.  Workload at N=1: BASELINE.json configs[1] -- the 128-window batch of
``inference.py --b 128`` on synthetic (200 reads x 90 columns) uint8 windows with random-init weights
(the reference-generated ``tests/golden/rand_seed1.pth``).  BASELINE.json's "200 pos x 30 reads" is
not executable by the reference (SURVEY.md section 0.3); the geometry here is the reference's.

Prints ONE JSON line (rank 0).  ``value`` = windows/s with inputs resident in HBM, device-timed;
``e2e`` = the same metric through ``RNN.predict_host`` (C ABI ``roko_b200_infer_host``) with pinned
HOST buffers, copies inside the timed region.  ``--impl reference`` times the reference's CPU
operator sequence (oracle/torch_port.py) on this box's host cores.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

READS, COLS, CLASSES = 200, 90, 5
WIN_BYTES = READS * COLS
STAGES = ["front", "proj0", "rec0", "proj1", "rec1", "proj2", "rec2", "head"]
# algorithmic FLOPs per window (SURVEY.md section 8d; fc1 one-hot factorised)
FLOPS = {"front": 90 * (200 * 100 + 2 * 100 * 50 * 12) + 2 * 90 * 50 * 100 * 10,
         "proj0": 2 * 90 * 768 * 500, "proj1": 2 * 90 * 768 * 256, "proj2": 2 * 90 * 768 * 256,
         "rec0": 2 * 90 * 768 * 128, "rec1": 2 * 90 * 768 * 128, "rec2": 2 * 90 * 768 * 128,
         "head": 2 * 90 * 256 * 5}
FLOPS_PER_WINDOW = sum(FLOPS.values())             # 214 813 440
ALG_BYTES_PER_WINDOW = READS * COLS + COLS         # 18 090: uint8 features in + uint8 labels out


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm_gbs": float(p["hbm_gbs"]), "bf16_tflops": float(p["bf16_tflops"]),
                "bf16_tflops_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])),
                "source": "measured"}
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self, windows=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, r in self.rows:
            if windows and not any(a <= ts <= b for a, b in windows):
                continue                                                # keep only samples taken inside a timed region
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for nm, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        busy = [v for v in sm if v > 0]
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dist_env():
    world = int(os.environ.get("WORLD_SIZE", "1"))
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), world


def host_cores():
    """CPUs this process may really use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:                       # cgroup v2
            quota, period = f.read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        try:                                                            # cgroup v1
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // p))
        except Exception:
            pass
    return max(1, n)


class CpuReference:
    """The reference's CPU operator sequence (oracle/torch_port.py) on this box's host cores.
    Every run is bounded by WALL TIME: a calibration probe picks sample sizes."""

    def __init__(self, threads=None):
        import torch
        from oracle.torch_port import TorchCpuPort
        self.torch = torch
        # MKL/oneDNN GEMMs of this size stop scaling well before 32 threads; more only oversubscribes
        self.threads = int(threads or min(host_cores(), 32))
        sd = torch.load(os.path.join(ROOT, "tests", "golden", "rand_seed1.pth"), map_location="cpu")
        self.port = TorchCpuPort(sd, threads=self.threads)
        self.gen = torch.Generator().manual_seed(1234)

    def windows(self, n):
        return self.torch.randint(0, 12, (n, READS, COLS), dtype=self.torch.uint8, generator=self.gen)

    def probe(self):
        """Seconds per window: best of three 16-window batches after one warm-up batch."""
        x = self.windows(16)
        self.port.predict(x)
        best = float("inf")
        for _ in range(3):
            t0 = time.perf_counter()
            self.port.predict(x)
            best = min(best, (time.perf_counter() - t0) / 16)
        return best

    def timed(self, steps, sample):
        x = self.windows(sample)
        t0 = time.perf_counter()
        for _ in range(steps):
            self.port.predict(x)
        dt = time.perf_counter() - t0
        return steps * sample / dt, dt


def cpu_baseline_bounded(budget_s=15.0, batch=128):
    ref = CpuReference()
    per_win = ref.probe()
    sample = int(max(1, min(batch, budget_s / 2 / per_win)))             # one batch <= half the budget
    steps = int(max(1, min(64, budget_s / (sample * per_win))))
    ref.timed(1, sample)
    wps, dt = ref.timed(steps, sample)
    return wps, ref.threads, f"{steps} x {sample} windows in {dt:.1f} s"


def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return
    batch, steps, warm = args.batch, args.steps, max(1, args.warmup)
    ref = CpuReference()
    per_win = ref.probe()
    # each step is a bounded sample of the batch so that W + K steps end within ~2 minutes
    budget = 120.0
    sample = int(max(1, min(batch, budget / (steps + warm) / per_win)))
    ref.timed(warm, sample)
    wps, dt = ref.timed(steps, sample)
    cores = ref.threads
    line = {
        "impl": "reference", "metric": "consensus_windows_per_sec", "value": wps, "unit": "windows/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": dt / steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"BASELINE configs[0]: reference CPU path, batch={batch}, windows (200 reads x 90 cols) uint8, "
                               "random-init .pth (tests/golden/rand_seed1.pth)", "batch": batch,
                   "sample_windows_per_step": sample, "host_cores_available": host_cores()},
        "cpu_baseline": {"value": wps, "unit": "windows/s", "cores": cores, "kind": "port",
                         "sample": f"{steps} steps x {sample} windows through the reference's stock-torch CPU operator "
                                   "sequence (oracle/torch_port.py; /root/reference is absent on the GPU box)"},
        "e2e": {"value": wps, "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


class StockTorchGpu:
    """Baseline B (BASELINE.md section 3): the reference's operator sequence on the SAME B200 through stock torch --
    embedding gather, permute + cuBLAS fc1/fc2, the cuDNN multi-layer bidirectional GRU, fc4, argmax
    (roko/rnn_model.py:46-59 after ``.to('cuda')``, roko/inference.py:91-116).  Library kernels only;
    none of this repo's kernels are on this path."""

    def __init__(self, state_dict, dev):
        import torch
        self.torch, self.dev = torch, dev
        self.sd = {k: v.detach().to(dev, torch.float32) for k, v in state_dict.items()}
        self.gru = torch.nn.GRU(500, 128, num_layers=3, batch_first=True, bidirectional=True).to(dev)
        own = self.gru.state_dict()
        for k in own:
            own[k].copy_(self.sd["gru." + k])
        self.gru.eval()
        self.gru.flatten_parameters()

    def predict(self, x_u8):
        torch, F, sd = self.torch, self.torch.nn.functional, self.sd
        x = x_u8.long()                                                       # inference.py:113
        h = F.embedding(x, sd["embedding.weight"]).permute((0, 2, 3, 1))      # rnn_model.py:47-48
        h = F.relu(F.linear(h, sd["fc1.weight"], sd["fc1.bias"]))             # :50
        h = F.relu(F.linear(h, sd["fc2.weight"], sd["fc2.bias"]))             # :53
        h, _ = self.gru(h.reshape(-1, 90, 500))                               # :56-57
        return torch.argmax(F.linear(h, sd["fc4.weight"], sd["fc4.bias"]), dim=2)   # :59, inference.py:116

    def windows_per_s(self, pool, batch, steps=None, min_s=0.4):
        """Device-timed steady-state throughput at `batch` windows per call over a pool of resident inputs:
        exactly `steps` calls, or groups of 8 calls until `min_s` seconds when `steps` is None."""
        torch = self.torch
        xs = pool.view(-1, READS, COLS)
        n = xs.shape[0] // batch
        with torch.no_grad():
            for i in range(3):
                self.predict(xs[(i % n) * batch:(i % n + 1) * batch])
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            done, ms = 0, 0.0
            while (done < steps) if steps else (ms < min_s * 1e3 and done < 2000):
                k = min(8, steps - done) if steps else 8
                e0.record()
                for i in range(k):
                    self.predict(xs[((done + i) % n) * batch:((done + i) % n + 1) * batch])
                e1.record()
                torch.cuda.synchronize()
                ms += e0.elapsed_time(e1)
                done += k
        return done * batch / (ms * 1e-3)


def run_torch_gpu(args):
    """bench.py --impl torch_gpu: baseline B as its own JSON line (same metric / config as the default arm)."""
    import torch
    rank, local_rank, world = dist_env()
    if rank != 0:
        return
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    sd = torch.load(os.path.join(ROOT, "tests", "golden", "rand_seed1.pth"), map_location="cpu")
    g = torch.Generator(device=dev).manual_seed(1234)
    pool = torch.randint(0, 12, (args.pool_batches, args.batch, READS, COLS), dtype=torch.uint8, device=dev, generator=g)
    stock = StockTorchGpu(sd, dev)
    wps = stock.windows_per_s(pool, args.batch, steps=args.steps)
    print(json.dumps({
        "impl": "torch_gpu", "metric": "consensus_windows_per_sec", "value": wps, "unit": "windows/s", "n_gpus": 1,
        "steps": args.steps, "warmup": 3, "ms_per_step": args.batch / wps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"BASELINE configs[1] geometry through STOCK torch on the GPU (cuBLAS + cuDNN GRU), batch={args.batch}",
                   "batch": args.batch, "tf32": bool(torch.backends.cuda.matmul.allow_tf32), "torch": torch.__version__},
        "gpu_launches": 0}), flush=True)


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from roko_b200 import _cabi
    from roko_b200 import dist as rdist
    from roko_b200.rnn_model import RNN, IN_SIZE, HIDDEN_SIZE, NUM_LAYERS
    from roko_b200.synth import structured_windows

    rank, local_rank, world = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl ours) needs a B200: the hot path is CUDA only, there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    batch, K, W, NS = args.batch, args.steps, max(args.streams, args.warmup), args.streams
    peaks = load_peaks()

    # ---- model: rank 0 loads the .pth, NCCL-broadcasts the weights ---------------------------------
    sd = torch.load(os.path.join(ROOT, "tests", "golden", "rand_seed1.pth"), map_location="cpu")
    model = RNN(IN_SIZE, HIDDEN_SIZE, NUM_LAYERS)
    if rank == 0:
        model.load_state_dict(sd)
    model = model.to(dev).eval().requires_grad_(False)
    bcast_bytes = rdist.broadcast_weights(model, src=0) if world > 1 else 0
    # throughput configuration: several batches in flight on different streams; the tensor-core recurrence
    # occupies 8 SMs per 128-window batch, so batches on other streams run beside it
    model.set_option("rec_tc_min", args.rec_tc_min)
    for name in ("proj", "rec", "front", "graphs"):
        v = getattr(args, name)
        if v is not None:
            model.set_option(name, v)

    # ---- parity gate before any timing, on the SAME kernels the timed loop runs: one full 128-window batch
    # (the reference class's own logits / labels, tests/golden/golden_b128_seed1.npz) through the same call ------
    gold = np.load(os.path.join(ROOT, "tests", "golden", "golden_b128_seed1.npz"))
    gx = structured_windows(128, seed=int(gold["seed"]))
    assert int(gx.astype(np.int64).sum()) == int(gold["x_crc"]), "synthetic generator drifted from the fixture"
    with torch.no_grad():
        lab, logit = model.predict(torch.from_numpy(gx).to(dev), return_logits=True)
    perr = float(np.abs(logit.cpu().numpy() - gold["logits"]).max())
    if perr > 1e-4 or not np.array_equal(lab.cpu().numpy(), gold["labels"]):
        raise SystemExit(f"parity gate failed on rank {rank}: max logit err {perr}")
    model.check_codes()

    # ---- synthetic pool, larger than L2 so no step re-reads its input from cache -------------------
    P = args.pool_batches

    def make_pool(r):
        g = torch.Generator(device=dev).manual_seed(1234 + r)
        return torch.randint(0, 12, (P, batch, READS, COLS), dtype=torch.uint8, device=dev, generator=g)

    pool = make_pool(rank)
    labels_all = torch.empty((K, batch, COLS), dtype=torch.uint8, device=dev)
    streams = [torch.cuda.Stream(device=dev) for _ in range(NS)]
    main = torch.cuda.current_stream(dev)

    def run_steps(n, out, src=None, first=0):
        """n steps (one per 128-window batch, NS batches in flight) over pool batches first, first + 1, ..."""
        src = pool if src is None else src
        for s in streams:
            s.wait_stream(main)
        for i in range(n):
            with torch.cuda.stream(streams[i % NS]):
                model.predict(src[(first + i) % P], out=out[i % out.shape[0]])
        for s in streams:
            main.wait_stream(s)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.12)
    with torch.no_grad():
        # the warm-up gives every stream at least one step: its workspace and CUDA graph are made outside the timed region
        run_steps(W, labels_all)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        # the timed region is exactly K steps between one CUDA-event pair, plus their label gather when N > 1; they start
        # at the pool batch after the warm-up's, so up to P - W steps read inputs no earlier step left in L2
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tw0 = time.perf_counter()
        e0.record(main)
        run_steps(K, labels_all, first=W)
        gathered = rdist.gather_labels(labels_all.view(K * batch, COLS), K * batch * world) if world > 1 else None
        e1.record(main)
        torch.cuda.synchronize()
        tw1 = time.perf_counter()
        if world > 1:
            dist.barrier()
        ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = K * batch * world / (ms * 1e-3)

    if args.dump_outputs and rank == 0:
        # the last timed step's labels: this rank's batch, or every rank's batch in rank order as gathered on rank 0
        last = gathered.view(world, K, batch, COLS)[:, K - 1].reshape(world * batch, COLS) if world > 1 else labels_all[K - 1]
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "labels.npy"), last.cpu().numpy().astype(np.float32))

    # ---- N > 1: what rank 0 gathered over NVLink must equal, byte for byte, what ONE GPU computes for every
    # rank's inputs (rank 0 regenerates each rank's seeded pool and replays that rank's timed steps) ----------
    shard_check = None
    if world > 1 and rank == 0:
        assert gathered is not None and gathered.shape == (K * batch * world, COLS)
        ok = True
        with torch.no_grad():
            for r in range(world):
                src = pool if r == 0 else make_pool(r)
                mine = torch.empty((K, batch, COLS), dtype=torch.uint8, device=dev)
                run_steps(K, mine, src=src, first=W)
                torch.cuda.synchronize()
                ok = ok and bool(torch.equal(mine.view(K * batch, COLS), gathered[r * K * batch:(r + 1) * K * batch]))
                del src
        if not ok:
            raise SystemExit("multi-GPU check failed: gathered labels differ from the single-GPU labels")
        shard_check = "gathered labels of every rank == single-GPU recomputation, byte for byte"

    # ---- e2e: pinned host windows -> labels on the host, through the public API ---------------------
    # K steps' inputs sit in pinned host memory; ONE predict_host call moves them to the device, runs the
    # path and brings the labels back.  Calls repeat until the region is >= min_region seconds.
    Kh = min(max(K, 512), max(1, (1280 << 20) // (batch * WIN_BYTES)))  # >= 512 batches per call (27 device passes), <= 1.25 GB pinned
    x_host = torch.empty((Kh * batch, READS, COLS), dtype=torch.uint8).pin_memory()
    for i0 in range(0, Kh, P):
        n = min(P, Kh - i0)
        x_host[i0 * batch:(i0 + n) * batch].copy_(pool[:n].view(n * batch, READS, COLS))
    y_host = torch.empty((Kh * batch, COLS), dtype=torch.uint8).pin_memory()
    torch.cuda.synchronize()
    model.predict_host(x_host[:min(Kh, 40) * batch], batch=batch, out=y_host[:min(Kh, 40) * batch])   # warm the slots
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    calls = 0
    while True:
        model.predict_host(x_host, batch=batch, out=y_host)
        calls += 1
        e2e_s = time.perf_counter() - t0
        stop = e2e_s >= args.min_region or calls >= 64
        if world > 1:                                                   # every rank makes the same number of calls
            t = torch.tensor([1.0 if stop else 0.0], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            stop = bool(t.item() > 0)
        if stop:
            break
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = calls * Kh * batch * world / e2e_s
    # clocks sampled inside the two timed regions (device-resident steps, end-to-end calls)
    clocks = sampler.stop([(tw0, tw1), (t0, t0 + e2e_s)]) if rank == 0 else None
    del x_host

    # ---- per-kernel device times (CUDA events between the kernels of the chain) -> roofline --------
    h = model._handle(dev)
    lib = h.lib
    ws = torch.empty(lib.roko_b200_workspace_bytes(batch), dtype=torch.uint8, device=dev)
    st = (ctypes.c_float * 8)()
    _cabi.check(lib.roko_b200_forward_timed(h.ptr, pool[0].data_ptr(), batch, labels_all[0].data_ptr(), ws.data_ptr(),
                                             ws.numel(), main.cuda_stream, 20, st))
    stage_ms = dict(zip(STAGES, [float(v) for v in st]))
    names = kernel_names(args, batch)
    kern_ms = {}
    for sname, v in stage_ms.items():
        kern_ms.setdefault(names[sname], []).append((sname, v))
    dom_kernel = max(kern_ms, key=lambda k: sum(v for _, v in kern_ms[k]))
    dom_stage = max(kern_ms[dom_kernel], key=lambda sv: sv[1])[0]
    dom_launch_ms = statistics.mean(v for _, v in kern_ms[dom_kernel])
    dom_flops = statistics.mean(FLOPS[s] for s, _ in kern_ms[dom_kernel]) * batch
    achieved_tf = dom_flops / (dom_launch_ms * 1e-3) / 1e12
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    dom_ctas = {"rec_h_kernel": 2 * ((batch + 31) // 32), "rec_tc_kernel": 2 * ((batch + 31) // 32),
                "rec_kernel": min(2 * ((batch + 1) // 2), sms), "front_kernel": min(batch, sms),
                "front_tc_kernel": min(batch, sms), "head_kernel": sms}.get(dom_kernel, sms)
    fp32 = ctypes.c_double()
    _cabi.check(lib.roko_b200_measure_fp32_peak(local_rank, ctypes.byref(fp32)))
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        traffic = tj.get(f"{dom_kernel}@B{batch}")
    except Exception:
        pass

    # ---- the same work coalesced: consecutive 128-window steps handed to the path as one device pass ---
    # (windows are independent; this is what predict_host / inference.py do internally)
    big = min(args.coalesce, P * batch)
    xb = pool.view(P * batch, READS, COLS)[:big]
    lb = torch.empty((big, COLS), dtype=torch.uint8, device=dev)
    ws_big = torch.empty(lib.roko_b200_workspace_bytes(big), dtype=torch.uint8, device=dev)
    st2 = (ctypes.c_float * 8)()
    _cabi.check(lib.roko_b200_forward_timed(h.ptr, xb.data_ptr(), big, lb.data_ptr(), ws_big.data_ptr(),
                                             ws_big.numel(), main.cuda_stream, 10, st2))
    big_ms = dict(zip(STAGES, [float(v) for v in st2]))
    big_total = sum(big_ms.values())
    big_names = kernel_names(args, big)
    big_kernels = {}
    for sname, v in big_ms.items():
        d = big_kernels.setdefault(big_names[sname], {"ms": 0.0, "flops": 0.0, "launches": 0})
        d["ms"] += v; d["flops"] += FLOPS[sname] * big; d["launches"] += 1
    for kname, d in big_kernels.items():
        # the fp16-split tensor kernels issue 3 MMAs per algorithmic product: that is the rate the tensor pipe actually sustains
        if kname.startswith(("proj_h", "rec_h", "proj_tc3", "rec_tc")):
            d["mma_tflops"] = 3 * d["flops"] / (d["ms"] * 1e-3) / 1e12
            d["mma_frac_of_bf16_tensor_peak"] = d["mma_tflops"] / (peaks["bf16_tflops_sustained"] / (2 if "tc" in kname else 1))
        d["tflops"] = d["flops"] / (d["ms"] * 1e-3) / 1e12
        d["frac_of_bf16_tensor_peak"] = d["tflops"] / peaks["bf16_tflops_sustained"]
        d["frac_of_fp32_ffma_peak"] = d["tflops"] / fp32.value if fp32.value else None
        del d["flops"]
    del ws_big

    # ---- baseline B: the stock torch operator sequence (cuBLAS + cuDNN GRU) on this same GPU ----------
    vs_library = None
    if rank == 0 and not args.no_library_baseline:
        try:
            stock = StockTorchGpu(sd, dev)
            lib128 = stock.windows_per_s(pool, batch)
            lib1024 = stock.windows_per_s(pool, 1024)
            vs_library = {"torch_gpu_windows_per_s": lib128, "torch_gpu_windows_per_s_b1024": lib1024,
                          "ratio": value / world / lib128, "ratio_vs_b1024": value / world / lib1024,
                          "note": "reference operator sequence through stock torch on this GPU (cuBLAS fp32 + cuDNN GRU), "
                                  "device-resident inputs, per-GPU; tf32=%s" % bool(torch.backends.cuda.matmul.allow_tf32)}
            del stock
        except Exception as ex:                                          # a library failure must not cost the bench line
            vs_library = {"unavailable": repr(ex)[:200]}

    if world > 1:
        dist.barrier()
    if rank == 0:
        line = {
            "metric": "consensus_windows_per_sec", "value": value, "unit": "windows/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "timed_region_s": ms * 1e-3,
            "config": {
                "workload": f"BASELINE configs[1]: batch={batch} synthetic windows (200 reads x 90 cols, uint8 codes 0..11) "
                            "per step on each GPU, random-init weights tests/golden/rand_seed1.pth, labels out (uint8)",
                "batch": batch, "windows_per_step_all_gpus": batch * world, "parallelism": f"dp{world}",
                "streams": NS,
                "timing": f"exactly {K} steps between one CUDA-event pair after {W} warm-up steps; ms_per_step = region / {K}",
                "e2e_note": "predict_host coalesces consecutive batches into device passes of <= 2368 windows "
                            "(windows are independent), so e2e can exceed the per-call batch-128 device number",
                "l2": f"step i reads batch ({W} + i) mod {P} of a {P * batch * WIN_BYTES / 1e6:.0f} MB pool (> 126 MB L2)",
                "collectives": ("ncclBroadcast weights %d B before timing; label all-gather of the timed steps inside the timed region" % bcast_bytes)
                               if world > 1 else "none (1 GPU)",
                "kernels": names,
            },
            "e2e": {"value": e2e_value, "unit": "windows/s", "h2d_bytes_per_step": batch * WIN_BYTES,
                    "d2h_bytes_per_step": batch * COLS, "api": "RNN.predict_host -> roko_b200_infer_host (pinned host buffers)",
                    "calls": calls, "windows_per_call": Kh * batch, "timed_region_s": e2e_s},
            "gpu_launches": K * 8,
            "clocks": clocks,
            "parity": {"batch128_max_abs_logit_err": perr, "batch128_labels_exact": True,
                       "fixture": "tests/golden/golden_b128_seed1.npz (reference class outputs), same kernels as the timed loop",
                       "multi_gpu": shard_check},
            "roofline": {"bound": "tensor", "kernel": dom_kernel, "stage": dom_stage, "achieved": achieved_tf,
                         "ctas_per_launch": dom_ctas, "sms": sms,
                         "frac_on_occupied_sms": achieved_tf / (peaks["bf16_tflops_sustained"] * min(dom_ctas, sms) / sms),
                         "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                         "frac": achieved_tf / peaks["bf16_tflops_sustained"], "traffic": traffic,
                         "peak_source": peaks["source"] + " bf16 dense, sustained (kernel timed inside the step)",
                         "note": "per-launch figure of one 128-window batch; algorithmic fp32 FLOPs (the tensor kernels spend 3 "
                                 "fp16 MMAs per product, so the MMA rate is 3x this); a launch of the tensor-core recurrence "
                                 "occupies only ctas_per_launch SMs while other batches run beside it; the whole-chip picture is "
                                 "coalesced.kernels"},
            "fp32": {"peak_tflops_measured": fp32.value, "kernel_frac": achieved_tf / fp32.value if fp32.value else None,
                     "path_tflops": value / world * FLOPS_PER_WINDOW / 1e12,
                     "path_frac": value / world * FLOPS_PER_WINDOW / 1e12 / fp32.value if fp32.value else None},
            "hbm": {"algorithmic_bytes_per_window": ALG_BYTES_PER_WINDOW, "achieved_gbs": value / world * ALG_BYTES_PER_WINDOW / 1e9,
                    "peak_gbs": peaks["hbm_gbs"], "frac": value / world * ALG_BYTES_PER_WINDOW / 1e9 / peaks["hbm_gbs"],
                    "note": "path is compute/latency bound (AI ~ 12 kFLOP/B); HBM fraction is <1 % by construction"},
            "stage_ms": stage_ms,
            "coalesced": {"windows_per_pass": big, "windows_per_s_per_gpu": big / (big_total * 1e-3), "ms_per_pass": big_total,
                          "stage_ms": big_ms, "kernels": big_kernels,
                          "path_tflops": big / (big_total * 1e-3) * FLOPS_PER_WINDOW / 1e12,
                          "path_frac_of_bf16_tensor_peak": big / (big_total * 1e-3) * FLOPS_PER_WINDOW / 1e12 / peaks["bf16_tflops_sustained"],
                          "note": "device-resident, one stream, consecutive steps fused into one pass (what predict_host does); "
                                  "TFLOP/s are algorithmic fp32 FLOPs: the tensor kernels spend 3 fp16 MMAs per product"},
            "vs_library": vs_library,
        }
        if world == 1 and not args.no_train:
            tms, _ = train_steps(dev, 128, 20, 3)
            line["training"] = {"windows_per_s": 128 / (tms * 1e-3), "ms_per_step": tms, "batch": 128,
                                "note": "roko train.py step (train-mode forward with dropout, cross-entropy, hand-written "
                                        "backward, Adam) on device-resident synthetic windows; see bench.py --mode train"}
        if world == 1 and not args.no_cpu_baseline:
            wps, cores, sample = cpu_baseline_bounded(15.0, batch)
            line["cpu_baseline"] = {"value": wps, "unit": "windows/s", "cores": cores, "kind": "port",
                                    "sample": sample + " through the reference's stock-torch CPU operator sequence "
                                              "(oracle/torch_port.py), time-bounded"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def kernel_names(args, nwin):
    """Which kernel runs each stage of the chain for a chunk of `nwin` windows under this run's options."""
    proj = {None: "proj_h_kernel", 4: "proj_h_kernel", 3: "proj_tc3_kernel", 0: "proj_kernel"}[args.proj]
    rec_tc = {None: "rec_h_kernel", 2: "rec_h_kernel", 1: "rec_tc_kernel"}[args.rec]
    if not (args.rec_tc_min and nwin >= args.rec_tc_min) or (rec_tc == "rec_tc_kernel" and nwin < 64):
        rec_tc = "rec_kernel"
    front = "front_kernel" if args.front == 0 else "front_tc_kernel"
    return {"front": front, "proj0": proj + "<512>", "proj1": proj + "<256>", "proj2": proj + "<256>",
            "rec0": rec_tc, "rec1": rec_tc, "rec2": rec_tc, "head": "head_kernel"}


def train_steps(dev, batch, steps, warmup, world=1, seed=0):
    """Reference training step (roko/train.py:41-55: train mode, zero_grad, forward, cross-entropy, backward,
    Adam lr 1e-4) on synthetic labelled windows resident on the device; gradients averaged over ranks with one
    flat all-reduce when world > 1.  Returns (ms per step from CUDA events, last loss)."""
    import torch
    import torch.nn.functional as F
    from roko_b200 import dist as rdist
    from roko_b200.rnn_model import RNN, IN_SIZE, HIDDEN_SIZE, NUM_LAYERS
    torch.manual_seed(seed)
    model = RNN(IN_SIZE, HIDDEN_SIZE, NUM_LAYERS).to(dev).train()
    if world > 1:
        rdist.broadcast_weights(model, src=0)
    opt = torch.optim.Adam(model.parameters(), lr=1e-4, fused=True)      # as roko_b200/train.py creates it
    g = torch.Generator(device=dev).manual_seed(77 + seed)
    pool = 8                                                   # 8 x 2.3 MB inputs; activations (1 GB) dwarf L2 anyway
    xs = torch.randint(0, 12, (pool, batch, READS, COLS), dtype=torch.uint8, device=dev, generator=g)
    ys = torch.randint(0, 5, (pool, batch, COLS), dtype=torch.int64, device=dev, generator=g)
    beg, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    loss = None
    for i in range(warmup + steps):
        if i == warmup:
            torch.cuda.synchronize()
            if world > 1:
                torch.distributed.barrier()
            beg.record()
        model.zero_grad()
        loss = F.cross_entropy(model(xs[i % pool]).transpose(1, 2), ys[i % pool])
        loss.backward()
        if world > 1:
            rdist.average_gradients(model)
        opt.step()
    end.record()
    torch.cuda.synchronize()
    return beg.elapsed_time(end) / steps, float(loss.item())


def run_train(args):
    """bench.py --mode train: BASELINE.json config 5 (training), weak scaling, one JSON line on rank 0."""
    import torch
    import torch.distributed as dist
    rank, local_rank, world = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --mode train needs a B200: the training kernels are CUDA only")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    K, W = args.steps, max(3, args.warmup)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms, loss = train_steps(dev, args.batch, K, W, world, seed=rank)
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        ms = float(t.item())
        print(json.dumps({
            "metric": "train_windows_per_s", "value": args.batch * world / (ms * 1e-3), "unit": "windows/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "roko train.py step: RNN(500,128,3) train mode (dropout 0.2), cross-entropy, backward, Adam 1e-4; "
                                   "x = (batch,200,90) u8 uniform codes, y uniform labels, device resident",
                       "batch_per_gpu": args.batch, "parallelism": f"dp{world}",
                       "collectives": "one flat 4.4 MB gradient all-reduce per step" if world > 1 else "none (1 GPU)"},
            "last_loss": loss, "clocks": clocks}), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mode", default="infer", choices=["infer", "train"],
                    help="infer: the north-star hot path (default); train: the training step")
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch_gpu"])
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--streams", type=int, default=12, help="batches in flight (one stream each); 12 measured best on B200: 8 -> 648 k, 12 -> 748 k, 16 -> 748 k windows/s")
    ap.add_argument("--rec-tc-min", type=int, default=64, help="windows from which the recurrence runs on tcgen05")
    ap.add_argument("--proj", type=int, default=None, help="projection kernel: 4 fp16 tcgen05 (default), 3 tf32 tcgen05, 0 FFMA")
    ap.add_argument("--rec", type=int, default=None, help="tensor-core recurrence: 2 fp16 (default), 1 tf32")
    ap.add_argument("--front", type=int, default=None, help="front end: 0 mma.sync stages, 1 tcgen05 stages (library default if unset)")
    ap.add_argument("--graphs", type=int, default=None, help="CUDA-graph replay of the chain: 1 on (default), 0 off")
    ap.add_argument("--min-region", type=float, default=0.5, help="repeat the end-to-end predict_host call until its timed region is this long (s)")
    ap.add_argument("--no-library-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--pool-batches", type=int, default=64)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--coalesce", type=int, default=2368, help="windows in the coalesced device pass (extra fields)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the labels of the last timed step to DIR/labels.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.mode != "infer"):
        ap.error("--dump-outputs writes the outputs of the inference path (--impl ours --mode infer)")
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "torch_gpu":
        run_torch_gpu(args)
    elif args.mode == "train":
        run_train(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
