#!/usr/bin/env python
"""Batch-128 throughput with many batches in flight, per launch geometry of the inference chain.

    python scripts/stream_throughput.py [--steps K] [--repeats R] [--front 2,4,8] [--proj 2,6,12] [--head 16,128,512]
                                        [--center 4,6,128] [--json OUT]

Runs bench.py's throughput loop in one process (12 streams, batch 128, a seeded pool of 64 batches, exactly K steps
between one CUDA-event pair) for geometry 0 (full-chip grids) and for geometry 1 with minima taken one knob at a time
around --center (windows per front_tc CTA, 128x256 tiles per proj_h CTA, rows per head block).  The settings are
visited round-robin, R times, so geometry 0 and 1 alternate and share whatever else the GPU is doing; each prints
its median windows/s and the spread (min..max).  Per setting it also prints each kernel's SM-time per window at
batch 128 (SMs held x stage time from roko_b200_forward_timed / windows; for the head, whose blocks share SMs, this
is an upper bound), the single-stream batch-128 latency, and checks that the timed steps' labels equal those of
geometry 0 byte for byte.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from bench import READS, COLS, STAGES, ClockSampler  # noqa: E402

BATCH, STREAMS, POOL = 128, 12, 64
TC_BM, GI_TILES_N, HEAD_ROWS_PER_BLOCK, HEAD_BLOCKS_PER_SM, REC_H_CTAS = 128, 3, 16, 8, 8


def grid_sizes(setting, sms, nwin=BATCH):
    """CTAs of each stage at `nwin` windows: the launchers' min(work, cap) with run_forward's caps (api.cu, model.h)."""
    def cap(units, per, full):
        return full if not setting["geometry"] else max(1, min(full, -(-units // per)))
    rows = nwin * COLS
    tiles = -(-rows // TC_BM) * GI_TILES_N
    front = min(nwin, cap(nwin, setting["geo_front"], sms))
    proj = min(tiles, cap(tiles, setting["geo_proj"], sms))
    head = min(-(-rows // HEAD_ROWS_PER_BLOCK), cap(rows, setting["geo_head"], HEAD_BLOCKS_PER_SM * sms))
    return {"front": front, "proj0": proj, "proj1": proj, "proj2": proj,
            "rec0": REC_H_CTAS, "rec1": REC_H_CTAS, "rec2": REC_H_CTAS, "head": head}


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [c.strip() for c in out.split(",")]))
    except Exception as ex:
        return {"unavailable": repr(ex)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3000)
    ap.add_argument("--warmup", type=int, default=24)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--center", default="4,6,128", help="geo_front,geo_proj,geo_head the one-knob sweeps vary around")
    ap.add_argument("--front", default="", help="geo_front values to sweep (comma separated)")
    ap.add_argument("--proj", default="", help="geo_proj values to sweep")
    ap.add_argument("--head", default="", help="geo_head values to sweep")
    ap.add_argument("--latency-calls", type=int, default=400)
    ap.add_argument("--json", default=None, help="also write every measurement to this file")
    args = ap.parse_args()

    import torch
    from roko_b200 import _cabi
    from roko_b200.rnn_model import RNN, IN_SIZE, HIDDEN_SIZE, NUM_LAYERS
    if not torch.cuda.is_available():
        raise SystemExit("stream_throughput.py needs a B200")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    sms = torch.cuda.get_device_properties(dev).multi_processor_count

    cf, cp, ch = (int(v) for v in args.center.split(","))
    settings = [dict(geometry=0, geo_front=cf, geo_proj=cp, geo_head=ch), dict(geometry=1, geo_front=cf, geo_proj=cp, geo_head=ch)]
    for key, vals in (("geo_front", args.front), ("geo_proj", args.proj), ("geo_head", args.head)):
        for v in (int(t) for t in vals.split(",") if t):
            s = dict(settings[1], **{key: v})
            if s not in settings:
                settings.append(s)

    sd = torch.load(os.path.join(ROOT, "tests", "golden", "rand_seed1.pth"), map_location="cpu")
    model = RNN(IN_SIZE, HIDDEN_SIZE, NUM_LAYERS)
    model.load_state_dict(sd)
    model = model.to(dev).eval().requires_grad_(False)
    model.set_option("rec_tc_min", 64)
    g = torch.Generator(device=dev).manual_seed(1234)
    pool = torch.randint(0, 12, (POOL, BATCH, READS, COLS), dtype=torch.uint8, device=dev, generator=g)
    K, W = args.steps, max(STREAMS, args.warmup)
    labels = torch.empty((K, BATCH, COLS), dtype=torch.uint8, device=dev)
    ref_labels = None
    streams = [torch.cuda.Stream(device=dev) for _ in range(STREAMS)]
    main_s = torch.cuda.current_stream(dev)

    def apply(s):
        for k, v in s.items():
            model.set_option(k, v)

    def run_steps(n, first=0):
        for st in streams:
            st.wait_stream(main_s)
        for i in range(n):
            with torch.cuda.stream(streams[i % STREAMS]):
                model.predict(pool[(first + i) % POOL], out=labels[i % K])
        for st in streams:
            main_s.wait_stream(st)

    info_before = gpu_info()
    sampler = ClockSampler(0)
    sampler.start()
    regions, wps = [], {i: [] for i in range(len(settings))}
    with torch.no_grad():
        for rep in range(args.repeats):
            for i, s in enumerate(settings):
                apply(s)
                run_steps(W)                                 # every stream captures its graph outside the timed region
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0 = time.perf_counter()
                e0.record(main_s)
                run_steps(K, first=W)
                e1.record(main_s)
                torch.cuda.synchronize()
                regions.append((t0, time.perf_counter()))
                wps[i].append(K * BATCH / (e0.elapsed_time(e1) * 1e-3))
                if ref_labels is None:
                    ref_labels = labels.clone()
                elif not torch.equal(labels, ref_labels):
                    raise SystemExit(f"labels of setting {s} differ from geometry 0")
    clocks = sampler.stop(regions)

    # per-kernel SM-time at batch 128 and single-stream latency, per setting
    h = model._handle(dev)
    lib = h.lib
    ws = torch.empty(lib.roko_b200_workspace_bytes(BATCH), dtype=torch.uint8, device=dev)
    lab1 = torch.empty((BATCH, COLS), dtype=torch.uint8, device=dev)
    results = []
    for i, s in enumerate(settings):
        apply(s)
        st = (ctypes.c_float * 8)()
        _cabi.check(lib.roko_b200_forward_timed(h.ptr, pool[0].data_ptr(), BATCH, lab1.data_ptr(), ws.data_ptr(),
                                                 ws.numel(), main_s.cuda_stream, 50, st))
        ctas = grid_sizes(s, sms)
        sm_us = {k: min(ctas[k], sms) * float(st[j]) * 1e3 / BATCH for j, k in enumerate(STAGES)}
        one = streams[0]
        with torch.no_grad(), torch.cuda.stream(one):
            for j in range(8):
                model.predict(pool[j], out=lab1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(one)
            for j in range(args.latency_calls):
                model.predict(pool[j % POOL], out=lab1)
            e1.record(one)
        torch.cuda.synchronize()
        lat_ms = e0.elapsed_time(e1) / args.latency_calls
        v = wps[i]
        results.append({"setting": s, "windows_per_s": v, "median": statistics.median(v), "min": min(v), "max": max(v),
                        "ctas_b128": ctas, "stage_ms_b128": dict(zip(STAGES, [float(t) for t in st])),
                        "sm_us_per_window_b128": sm_us, "sm_us_per_window_sum": sum(sm_us.values()),
                        "single_stream_ms_b128": lat_ms})

    base = results[0]["median"]
    print(f"gpu: {info_before}  sampled during the timed regions: {clocks}")
    print(f"{K} steps x {BATCH} windows, {STREAMS} streams, {args.repeats} repeats per setting, round-robin; labels equal "
          f"to geometry 0 in every timed region")
    print(f"{'geometry':>8} {'front':>5} {'proj':>4} {'head':>4} | {'median k/s':>10} {'min..max k/s':>15} {'vs g0':>6} | "
          f"{'CTAs f/p/h':>11} | SM-us/window front proj(x3) rec(x3) head = sum | 1-stream ms")
    for r in results:
        s, c, u = r["setting"], r["ctas_b128"], r["sm_us_per_window_b128"]
        proj = u["proj0"] + u["proj1"] + u["proj2"]
        rec = u["rec0"] + u["rec1"] + u["rec2"]
        print(f"{s['geometry']:>8} {s['geo_front']:>5} {s['geo_proj']:>4} {s['geo_head']:>4} | {r['median'] / 1e3:>10.1f} "
              f"{r['min'] / 1e3:>7.1f}..{r['max'] / 1e3:<7.1f} {r['median'] / base - 1:>+6.1%} | "
              f"{c['front']:>3}/{c['proj0']:>3}/{c['head']:>3} | {u['front']:5.1f} {proj:5.1f} {rec:5.1f} {u['head']:5.1f} "
              f"= {r['sm_us_per_window_sum']:5.1f} | {r['single_stream_ms_b128']:.3f}")
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump({"gpu": info_before, "gpu_after": gpu_info(), "clocks": clocks, "steps": K, "batch": BATCH,
                       "streams": STREAMS, "repeats": args.repeats, "sms": sms, "results": results}, f, indent=1)


if __name__ == "__main__":
    main()
