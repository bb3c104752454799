#!/usr/bin/env python
"""Benchmark of the stereo-matching hot path (BASELINE.json: disparity Mpix/s and cost-volume
Gvoxel/s on 1024x1024 rectified tiles, disp_range 128, census 5x5 + 8-path MGM, `mgm` flags of s2p).

    python bench.py --gpus N --steps K --warmup W              # our CUDA engine
    python bench.py --impl reference --gpus N --steps K ...    # the reference's CPU `mgm` on host cores
    python bench.py --steps K --dump-outputs DIR               # + the last timed step's outputs as DIR/*.npy, to compare builds

A "step" = one pass of the hot path over a batch of `--tiles` synthetic rectified pairs per GPU.
`value`  : whole-job Mpix/s with the pairs already resident in HBM (device pointers through
           s2pb_mgm_device, CUDA-event timed on the launching streams, max over ranks).
`e2e`    : the same metric through the reference-facing C-ABI call with HOST buffers
           (s2pb_mgm_batch from page-locked host buffers: H2D, kernels, D2H every step).
`roofline`: the 8-path aggregation kernel, algorithmic bytes (SURVEY.md section 8d: 12 B per voxel
           per path = 192 B per left-reference voxel for the two views) / its CUDA-event duration.
`cpu_baseline`: the reference's own `mgm` binary (oracle/_ref, built from the reference sources)
           on a bounded sample of the same workload, on this box's host cores.
`outputs_verified`: every output tile of the last timed step (8 tiles in flight) and of the last end-to-end step is
           compared bit for bit with a serial re-run of the same tile.
`extra_configs`: the other BASELINE.json configurations and the rest of the hot path, each with value / e2e / roofline /
           cpu_baseline: C3 (`mgm_multi`, 256 labels), C4 (a FIXED queue of 256 tiles 1026x1026x192 pulled dynamically by
           the ranks: strong scaling), C5 (tri-stereo: two pairs per tile + fusion.merge_n), C2 with 5 % no-data borders,
           and the rectification warp.
Tiles are independent: with N GPUs each rank processes its own tiles, no data-path collective.
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

METRIC = "disparity_throughput_1024x1024x128_mgm"
UNIT = "Mpix/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--tiles", type=int, default=16, help="tiles per GPU per step")
    ap.add_argument("--size", type=int, default=1024)
    ap.add_argument("--dmin", type=int, default=-64)
    ap.add_argument("--dmax", type=int, default=63)
    ap.add_argument("--slots", type=int, default=8, help="tiles in flight per GPU (one 8.5 GiB workspace each at the default shape)")
    ap.add_argument("--cpu-procs", type=int, default=0, help="concurrent reference processes (0 = calibrate: all host cores, 1/2, 1/4)")
    ap.add_argument("--cpu-rows", type=int, default=32, help="rows of the CPU sample strips")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra configurations (C3, C4, C5, no-data, warp)")
    ap.add_argument("--only-extra", default="", help="comma-separated subset of the extra configurations to run")
    ap.add_argument("--nan-border", type=float, default=0.0,
                    help="fraction of the tile width turned into no-data strips (0 = the BASELINE workload; > 0 exercises the "
                         "no-data sentinel range, which can widen the right view's slab: DESIGN.md, limits)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the disparity, confidence and rejection mask of the last device-resident step "
                         "(rank 0's tiles) as DIR/{disp,conf,mask}.npy, float32 of shape (tiles, H, W), and DIR/{disp,conf}_valid.npy "
                         "(1 where the output is finite, 0 where it is NaN = no match; the value itself is then written as 0); above "
                         "%d MB in all, the same seeded sample of pixels of each, flattened in (tile, row, column) order" % (DUMP_BYTES // 10 ** 6))
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(torch, out_dir, named):
    """Write the named lists of (H, W) device tensors to out_dir/<name>.npy as float32: whole when they fit DUMP_BYTES together,
    else each at the same seeded sample of flat indices.  Every file holds finite values only: a floating-point output is written
    with its non-finite values (NaN marks a pixel without a disparity) set to 0, beside <name>_valid.npy, 1 where it is finite.
    -> description for the JSON line."""
    os.makedirs(out_dir, exist_ok=True)
    first = next(iter(named.values()))
    nfiles = sum(2 if t[0].is_floating_point() else 1 for t in named.values())
    total = sum(t.numel() for t in first)
    n = min(total, (DUMP_BYTES - 4096 * nfiles) // (4 * nfiles))       # 4096: room for the .npy headers
    idx = None
    if n < total:
        rng = np.random.default_rng(0)
        idx = torch.from_numpy(np.sort(rng.choice(total, size=n, replace=False))).to(first[0].device)
    names = []
    for name, tensors in named.items():
        x = torch.stack(tensors)
        x = x if idx is None else x.reshape(-1)[idx]
        out = {name: x.float()}
        if x.is_floating_point():
            ok = torch.isfinite(x)
            out = {name: torch.where(ok, x, torch.zeros_like(x)).float(), name + "_valid": ok.float()}
        for k, v in out.items():
            np.save(os.path.join(out_dir, k + ".npy"), v.cpu().numpy())
            names.append(k)
    return {"dir": out_dir, "names": sorted(names), "dtype": "float32",
            "sampled": None if idx is None else "%d of %d pixels per output, numpy default_rng(0) choice without replacement, sorted" % (n, total)}


def config(a, world):
    return {
        "workload": "%ssingle %dx%d rectified tile, disp_range=%d, census5x5 + 8-path MGM "
                    "(s2p algo 'mgm': TSGM=3, P1=8, P2=32, vfit, MEDIAN=1, LR check), %d tiles per GPU per step" % (
                        "BASELINE configs[1]: " if (a.size, a.dmin, a.dmax) == (1024, -64, 63) else "", a.size, a.size,
                        a.dmax - a.dmin + 1, a.tiles),
        "tile": [a.size, a.size], "dmin": a.dmin, "dmax": a.dmax, "labels": a.dmax - a.dmin + 1,
        "tiles_per_gpu_per_step": a.tiles, "tiles_in_flight": a.slots, "parallelism": "tile-shard x%d" % world,
        "nan_border": a.nan_border,
        "l2": "per-tile working set %.1f GiB (8 float path volumes per view) >> 126 MB L2; inputs differ per tile" % (
            2 * 8 * 4.0 * a.size * a.size * (32 * ((a.dmax - a.dmin + 32) // 32)) / 2 ** 30 * 1.0625),
    }


# ----------------------------------------------------------------------------- clocks

class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def window(self, t0, t1):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        sm, reasons = [], set()
        for t, line in self.rows:
            if t < t0 or t > t1:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0]))
                out["sm_max_mhz"] = float(f[1])
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out["sm_mhz"] = float(np.median(sm))
        out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        return out

    def stop(self):
        if self.proc:
            self.proc.terminate()


# ----------------------------------------------------------------------------- reference CPU arm

def cpu_reference_step(strips, dmin, dmax, procs):
    """Run `procs` single-thread reference `mgm` processes concurrently (s2p's deployment mode:
    one process per tile, OMP_NUM_THREADS=1, s2p/config.py:46), one strip each.  -> seconds."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle as O
    P = O.mgm_params()
    t0 = time.perf_counter()
    with ThreadPoolExecutor(procs) as ex:
        list(ex.map(lambda rs: O.run_ref(rs[0], rs[1], dmin, dmax, P, threads=1), strips))
    return time.perf_counter() - t0


def make_strips(a, procs, base_tiles=None):
    from s2p_b200.synth import make_pair
    rows = min(a.cpu_rows, a.size)
    tiles = base_tiles or [make_pair(a.size, a.size, a.dmin, a.dmax, seed=s)[:2] for s in range(min(procs, 4))]
    strips = []
    for k in range(procs):
        ref, sec = tiles[k % len(tiles)]
        r0 = (k // len(tiles) * rows) % max(1, a.size - rows + 1)
        strips.append((ref[r0:r0 + rows], sec[r0:r0 + rows]))
    return strips, rows


def cpu_proc_candidates(a):
    """Process counts to try: the reference is memory-bound with many concurrent single-thread processes, so
    'all host threads' is not always its fastest deployment -- the best of (all, 1/2, 1/4 of the cores) is used."""
    n = os.cpu_count() or 1
    if a.cpu_procs > 0:
        return [a.cpu_procs]
    return sorted({n, max(1, n // 2), max(1, n // 4)}, reverse=True)


def cpu_best(a, base_tiles=None):
    """-> (Mpix/s, procs, rows, seconds, strips) of the fastest candidate, one step each."""
    best = None
    for procs in cpu_proc_candidates(a):
        strips, rows = make_strips(a, procs, base_tiles=base_tiles)
        secs = cpu_reference_step(strips, a.dmin, a.dmax, procs)
        mpix = procs * rows * a.size / secs / 1e6
        if best is None or mpix > best[0]:
            best = (mpix, procs, rows, secs, strips)
    return best


def run_reference(a, rank, world):
    if rank != 0:
        return
    from oracle import oracle as O
    if not O.have_ref():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/mgm not built (make -C oracle ref)"}))
        return
    _, procs, rows, _, strips = cpu_best(a)          # calibration doubles as warm-up
    for _ in range(max(0, a.warmup - len(cpu_proc_candidates(a)))):
        cpu_reference_step(strips, a.dmin, a.dmax, procs)
    t = [cpu_reference_step(strips, a.dmin, a.dmax, procs) for _ in range(a.steps)]
    total = sum(t)
    pix = procs * rows * a.size * a.steps
    val = pix / total / 1e6
    D = a.dmax - a.dmin + 1
    sample = "%d strips of %dx%d px, %d labels, one single-thread reference `mgm` process each (OMP_NUM_THREADS=1), PFM I/O included" % (
        procs, a.size, rows, D)
    # calibration of the strip sample: ONE full tile through one single-thread process (what one s2p worker does)
    full = None
    if (a.size, a.dmax - a.dmin + 1) == (1024, 128) and not a.no_extra:
        from s2p_b200.synth import make_pair
        r_, s_, _ = make_pair(a.size, a.size, a.dmin, a.dmax, seed=0)
        t0 = time.perf_counter()
        O.run_ref(r_, s_, a.dmin, a.dmax, O.mgm_params(), threads=1)
        dt = time.perf_counter() - t0
        full = {"tile": [a.size, a.size], "seconds": dt, "mpix_per_s_per_process": a.size * a.size / dt / 1e6,
                "strip_mpix_per_s_per_process": val / procs,
                "note": "one single-thread process alone on the box; the strips ran %d processes concurrently" % procs}
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1e3 * total / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": config(a, world), "gvoxel_per_s": val * D / 1e3,
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": procs, "kind": "reference", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "full_tile_calibration": full,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------- our arm

def run_ours(a, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from s2p_b200.engine import Engine, default_params
    from s2p_b200.synth import make_pair

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    W = H = a.size
    D = a.dmax - a.dmin + 1
    B = a.tiles
    p = default_params("mgm")
    eng = Engine(local_rank)
    nslots = max(1, min(a.slots, B))
    eng.reserve(nslots, W, H, D)

    # synthetic rectified pairs, distinct per tile and per rank (seed = global tile id)
    pairs = [make_pair(H, W, a.dmin, a.dmax, seed=rank * B + t, nan_border=a.nan_border)[:2] for t in range(B)]
    d_ref = [torch.from_numpy(r).to(dev) for r, _ in pairs]
    d_sec = [torch.from_numpy(s).to(dev) for _, s in pairs]
    d_disp = [torch.empty((H, W), dtype=torch.float32, device=dev) for _ in range(B)]
    d_conf = [torch.empty((H, W), dtype=torch.float32, device=dev) for _ in range(B)]
    d_mask = [torch.empty((H, W), dtype=torch.uint8, device=dev) for _ in range(B)]
    streams = [torch.cuda.Stream(device=dev) for _ in range(nslots)]
    main = torch.cuda.current_stream(dev)

    # The tile queue of a step is spread over `nslots` workspaces, each with its own stream; consecutive steps keep
    # the queue full (a workspace's stream orders its own tiles), the streams are joined where the timed region ends.
    def fork():
        ev = torch.cuda.Event()
        ev.record(main)
        for st in streams:
            st.wait_event(ev)

    def join():
        for st in streams:
            ev = torch.cuda.Event()
            ev.record(st)
            main.wait_event(ev)

    def device_step():
        for t in range(B):
            sl = t % nslots
            eng.mgm_device(sl, d_ref[t].data_ptr(), d_sec[t].data_ptr(), W, H, a.dmin, a.dmax, p, d_disp[t].data_ptr(),
                           d_conf[t].data_ptr(), d_mask[t].data_ptr(), 0, nodata_hint=(2 if a.nan_border > 0 else 0), stream=streams[sl].cuda_stream)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sampler = ClockSampler(local_rank) if rank == 0 else None

    # ---- device-resident arm
    fork()
    for _ in range(max(3, a.warmup)):
        device_step()
    join()
    barrier()
    l0 = eng.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tw0 = time.perf_counter()
    e0.record(main)
    fork()
    for _ in range(a.steps):
        device_step()
    join()
    e1.record(main)
    barrier()
    tw1 = time.perf_counter()
    launches = eng.kernel_launches() - l0
    ms = max_over_ranks(e0.elapsed_time(e1))
    dumped = None
    if a.dump_outputs and rank == 0:
        dumped = dump_outputs(torch, a.dump_outputs, {"disp": d_disp, "conf": d_conf, "mask": d_mask})
    # stage durations of the LAST tile of each workspace while the tiles overlap (diagnostic: how much the
    # memory-bound WTA stretches when it shares the SMs with the next tile's aggregation)
    overlapped = {}
    try:
        per_slot = [eng.last_timings(s) for s in range(len(streams))]
        overlapped = {k: float(np.mean([t[k] for t in per_slot])) for k in per_slot[0]}
    except Exception:
        pass
    pix_step = world * B * W * H
    value = pix_step * a.steps / (ms * 1e-3) / 1e6

    # every output tile of the last timed step (produced with `nslots` tiles in flight, WTA of one tile overlapping the
    # aggregation of the next) against a serial re-run of the same tile on one workspace: bit for bit
    valid = float(torch.isfinite(d_disp[0]).float().mean().item())
    chk = (torch.empty((H, W), dtype=torch.float32, device=dev), torch.empty((H, W), dtype=torch.float32, device=dev),
           torch.empty((H, W), dtype=torch.uint8, device=dev))
    hint = 2 if a.nan_border > 0 else 0
    bits = lambda t: t.view(torch.int32) if t.dtype == torch.float32 else t
    verified_device = True
    for t in range(B):
        eng.mgm_device(0, d_ref[t].data_ptr(), d_sec[t].data_ptr(), W, H, a.dmin, a.dmax, p, chk[0].data_ptr(), chk[1].data_ptr(),
                       chk[2].data_ptr(), 0, nodata_hint=hint, stream=streams[0].cuda_stream)
        streams[0].synchronize()
        ok = all(bool(torch.equal(bits(x), bits(y))) for x, y in zip(chk, (d_disp[t], d_conf[t], d_mask[t])))
        verified_device = verified_device and ok

    # ---- end-to-end arm: host buffers through the C ABI
    # host buffers are page-locked (torch pinned tensors viewed as numpy): the library DMAs from / to them directly
    keep = []

    def pinned(arr):
        t = torch.from_numpy(np.ascontiguousarray(arr)).pin_memory()
        keep.append(t)
        return t.numpy()
    refs = [pinned(r) for r, _ in pairs]
    secs = [pinned(s) for _, s in pairs]
    outs = ([pinned(np.empty((H, W), np.float32)) for _ in pairs], [pinned(np.empty((H, W), np.float32)) for _ in pairs],
            [pinned(np.empty((H, W), np.uint8)) for _ in pairs])
    for _ in range(max(1, min(3, a.warmup))):
        eng.mgm_batch(refs, secs, a.dmin, a.dmax, p, out=outs)
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        out = eng.mgm_batch(refs, secs, a.dmin, a.dmax, p, out=outs)
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e = pix_step * a.steps / e2e_s / 1e6
    h2d = B * 2 * W * H * 4
    d2h = B * (2 * W * H * 4 + W * H)
    # the end-to-end outputs of the last step against the device-resident ones (same inputs, other entry point)
    verified_e2e = all(np.array_equal(outs[0][t].view(np.int32), d_disp[t].cpu().numpy().view(np.int32)) and
                       np.array_equal(outs[1][t].view(np.int32), d_conf[t].cpu().numpy().view(np.int32)) and
                       np.array_equal(outs[2][t], d_mask[t].cpu().numpy()) for t in range(B))
    verified = verified_device and verified_e2e
    if world > 1:
        tv = torch.tensor([1.0 if verified else 0.0], device=dev)
        dist.all_reduce(tv, op=dist.ReduceOp.MIN)
        verified = bool(tv.item() > 0.5)

    # ---- roofline of the dominant kernel: serial launches on one stream, the library's own CUDA events
    agg_ms, tot_ms, stage = [], [], {}
    for k in range(max(3, min(a.steps, 10))):
        t = k % B
        eng.mgm_device(0, d_ref[t].data_ptr(), d_sec[t].data_ptr(), W, H, a.dmin, a.dmax, p, d_disp[t].data_ptr(),
                       d_conf[t].data_ptr(), d_mask[t].data_ptr(), 0, nodata_hint=(2 if a.nan_border > 0 else 0), stream=streams[0].cuda_stream)
        streams[0].synchronize()
        tm = eng.last_timings(0)
        agg_ms.append(tm["aggregate"])
        tot_ms.append(tm["total"])
        stage = tm
    agg = float(np.mean(agg_ms[1:]))
    alg_bytes = 192.0 * W * H * D          # 12 B/voxel/path x 8 paths x 2 views (SURVEY.md 8d)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = alg_bytes / (agg * 1e-3) / 1e9
    traffic, traffic_src = None, "not captured for this shape"
    if (W, H, D) == (1024, 1024, 128):      # the committed ncu capture is of this configuration
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["aggregate_kernel"]
            traffic = float(tj["bytes"])
            traffic_src = "profiles/traffic.json: %s" % tj.get("source", tj.get("capture", "ncu dram__bytes_read + dram__bytes_write per launch"))
        except (OSError, ValueError, KeyError):
            traffic = None
    roofline = {"bound": "hbm", "kernel": "aggregate_kernel (8 passes x 2 views, one persistent launch)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s",
                "traffic": traffic, "traffic_source": traffic_src,
                "frac_of_peak_on_real_traffic": (traffic / (agg * 1e-3) / 1e9 / peak) if traffic else None,
                "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": agg,
                "tile_ms_serial": float(np.mean(tot_ms[1:])), "stage_ms": stage,
                "stage_ms_overlapped": overlapped, "how": "serial single-tile launches after the timed region, CUDA events recorded by the library on the launching stream"}

    clocks = None
    if sampler:
        clocks = sampler.window(tw0, tw1)
        sampler.stop()

    # ---- CPU baseline beside it (rank 0, N=1 only): the reference binary on a bounded sample
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu:
        from oracle import oracle as O
        if O.have_ref():
            mpix, procs, rows, secs_cpu, _ = cpu_best(a, base_tiles=pairs[:4])
            cpu = {"value": mpix, "unit": UNIT, "cores": procs, "kind": "reference",
                   "sample": "%d strips of %dx%d px, %d labels, one single-thread reference `mgm` process each "
                             "(OMP_NUM_THREADS=1, the way s2p deploys it), %.1f s wall; fastest of %s concurrent processes on %d host threads"
                             % (procs, W, rows, D, secs_cpu, cpu_proc_candidates(a), os.cpu_count() or 1)}
        else:
            t0 = time.perf_counter()
            O.port.mgm(pairs[0][0][:64], pairs[0][1][:64], a.dmin, a.dmax, O.mgm_params())
            dt = time.perf_counter() - t0
            cpu = {"value": 64 * W / dt / 1e6, "unit": UNIT, "cores": min(8, os.cpu_count() or 1), "kind": "port",
                   "sample": "one %dx64 strip through oracle/liboracle.so (OpenMP over the 8 passes)" % W}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(3, a.warmup),
            "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": config(a, world), "gvoxel_per_s": value * D / 1e3,
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "timer": "host wall clock around the synchronised region, max over ranks; page-locked host buffers on both sides",
                    "gvoxel_per_s": e2e * D / 1e3},
            "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
            "valid_fraction_tile0": valid, "outputs_verified": verified,
            "outputs_verified_how": "all %d tiles of the last timed step (%d in flight) and of the last end-to-end step, bit for bit "
                                    "against a serial re-run of each tile (disparity, confidence, mask)" % (B, nslots),
            "dumped_outputs": dumped,
        }
    # ---- the other configurations (every rank takes part; rank 0 reports)
    extras = {}
    if not a.no_extra:
        del d_disp, d_conf, d_mask, chk, keep, refs, secs, outs
        torch.cuda.empty_cache()
        ctx = dict(a=a, eng=eng, rank=rank, world=world, dev=dev, torch=torch, dist=dist, barrier=barrier, max_over_ranks=max_over_ranks,
                   peak=peak, cpu=(rank == 0 and world == 1 and not a.no_cpu))
        only = [x for x in a.only_extra.split(",") if x]
        for name, fn in EXTRA:
            if only and name not in only:
                continue
            if world > 1 and name not in MULTI_RANK_EXTRA:      # the single-GPU configurations are reported by the N = 1 run
                continue
            try:
                extras[name] = fn(ctx)
            except Exception as e:       # an extra configuration must never cost the headline line
                extras[name] = {"error": "%s: %s" % (type(e).__name__, e)}
    if rank == 0:
        line["extra_configs"] = extras
        print(json.dumps(line))
    eng.close()
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------- the other configurations

def _pin(torch, keep, arr):
    t = torch.from_numpy(np.ascontiguousarray(arr)).pin_memory()
    keep.append(t)
    return t.numpy()


def _cpu_sample(binary, tiles, dmin, dmax, params, procs):
    """`procs` single-thread reference processes at once, one sample tile each -> (Mpix/s, seconds)"""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle as O
    t0 = time.perf_counter()
    with ThreadPoolExecutor(procs) as ex:
        list(ex.map(lambda rs: O.run_ref(rs[0], rs[1], dmin, dmax, params, threads=1, binary=binary), tiles))
    dt = time.perf_counter() - t0
    return sum(r.shape[0] * r.shape[1] for r, _ in tiles) / dt / 1e6, dt


def _matcher_config(ctx, algo, W, H, dmin, dmax, B, steps, nslots, nan_border=0.0, label=""):
    """One matcher configuration, both arms: device-resident (CUDA events) and end to end through s2pb_mgm_batch with
    page-locked host buffers.  -> dict(value, e2e, roofline, ...)"""
    torch, eng, a = ctx["torch"], ctx["eng"], ctx["a"]
    from s2p_b200.engine import default_params
    from s2p_b200.synth import make_pair
    dev, rank, world = ctx["dev"], ctx["rank"], ctx["world"]
    D = dmax - dmin + 1
    p = default_params(algo)
    pairs = [make_pair(H, W, dmin, dmax, seed=1000 + rank * B + t, nan_border=nan_border)[:2] for t in range(B)]
    multi = algo != "mgm"
    # mgm_multi reads a label hull back at every pyramid level, so a tile's enqueue blocks its host thread: tiles go in flight from
    # one host thread per workspace (here; s2pb_mgm_batch does the same inside the library), at most 4 (13 GiB of volumes each)
    nslots = max(1, min(4, nslots, B)) if multi else max(1, min(nslots, B))
    if not multi:
        eng.reserve(nslots, W, H, D + (1 if nan_border > 0 else 0))
    d_ref = [torch.from_numpy(r).to(dev) for r, _ in pairs]
    d_sec = [torch.from_numpy(s).to(dev) for _, s in pairs]
    d_out = [(torch.empty((H, W), dtype=torch.float32, device=dev), torch.empty((H, W), dtype=torch.float32, device=dev),
              torch.empty((H, W), dtype=torch.uint8, device=dev)) for _ in range(B)]
    streams = [torch.cuda.Stream(device=dev) for _ in range(nslots)]
    main = torch.cuda.current_stream(dev)
    hint = 2 if nan_border > 0 else 0

    def one_tile(t):
        sl = t % nslots
        eng.mgm_device(sl, d_ref[t].data_ptr(), d_sec[t].data_ptr(), W, H, dmin, dmax, p, d_out[t][0].data_ptr(), d_out[t][1].data_ptr(),
                       d_out[t][2].data_ptr(), 0, nodata_hint=hint, stream=streams[sl].cuda_stream)

    def device_step():
        if multi and nslots > 1:       # one host thread per workspace (ctypes releases the GIL during the call)
            from concurrent.futures import ThreadPoolExecutor
            with ThreadPoolExecutor(nslots) as ex:
                list(ex.map(lambda sl: [one_tile(t) for t in range(sl, B, nslots)], range(nslots)))
        else:
            for t in range(B):
                one_tile(t)

    def fork():
        ev = torch.cuda.Event(); ev.record(main)
        for st in streams:
            st.wait_event(ev)

    def join():
        for st in streams:
            ev = torch.cuda.Event(); ev.record(st); main.wait_event(ev)

    fork(); device_step(); join()
    ctx["barrier"]()
    l0 = eng.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(main); fork()
    for _ in range(steps):
        device_step()
    join(); e1.record(main)
    ctx["barrier"]()
    ms = ctx["max_over_ranks"](e0.elapsed_time(e1))
    launches = eng.kernel_launches() - l0
    pix = world * B * W * H * steps
    value = pix / (ms * 1e-3) / 1e6
    keep = []
    refs = [_pin(torch, keep, r) for r, _ in pairs]
    secs = [_pin(torch, keep, s) for _, s in pairs]
    outs = ([_pin(torch, keep, np.empty((H, W), np.float32)) for _ in pairs], [_pin(torch, keep, np.empty((H, W), np.float32)) for _ in pairs],
            [_pin(torch, keep, np.empty((H, W), np.uint8)) for _ in pairs])
    eng.mgm_batch(refs, secs, dmin, dmax, p, out=outs)
    ctx["barrier"]()
    t0 = time.perf_counter()
    for _ in range(steps):
        eng.mgm_batch(refs, secs, dmin, dmax, p, out=outs)
    ctx["barrier"]()
    e2e_s = ctx["max_over_ranks"](time.perf_counter() - t0)
    e2e = pix / e2e_s / 1e6
    same = all(np.array_equal(outs[0][t].view(np.int32), d_out[t][0].cpu().numpy().view(np.int32)) and
               np.array_equal(outs[1][t].view(np.int32), d_out[t][1].cpu().numpy().view(np.int32)) for t in range(B))
    res = {"workload": label, "tile": [W, H], "labels": D, "algo": algo, "tiles_per_gpu_per_step": B, "steps": steps, "tiles_in_flight": nslots,
           "metric": "disparity Mpix/s", "value": value, "unit": UNIT, "ms_per_tile": ms / (B * steps), "gvoxel_per_s": value * D / 1e3,
           "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": B * 2 * W * H * 4, "d2h_bytes_per_step": B * (2 * W * H * 4 + W * H)},
           "gpu_launches": int(launches), "e2e_equals_device_outputs": bool(same), "scaling": "weak", "nan_border": nan_border}
    if not multi:
        agg = []
        for k in range(4):
            t = k % B
            eng.mgm_device(0, d_ref[t].data_ptr(), d_sec[t].data_ptr(), W, H, dmin, dmax, p, d_out[t][0].data_ptr(), d_out[t][1].data_ptr(),
                           d_out[t][2].data_ptr(), 0, nodata_hint=hint, stream=streams[0].cuda_stream)
            streams[0].synchronize()
            agg.append(eng.last_timings(0))
        am = float(np.mean([x["aggregate"] for x in agg[1:]]))
        alg = 192.0 * W * H * D
        res["roofline"] = {"bound": "hbm", "kernel": "aggregate_kernel", "achieved": alg / (am * 1e-3) / 1e9, "peak": ctx["peak"], "unit": "GB/s",
                           "frac": alg / (am * 1e-3) / 1e9 / ctx["peak"], "kernel_ms": am, "algorithmic_bytes_per_launch": alg, "traffic": None,
                           "stage_ms": agg[-1]}
    else:
        # per-tile algorithmic bytes of mgm_multi are data dependent (per-pixel ranges); the whole-tile figure below uses the
        # dense 216 B / voxel of SURVEY.md 8d on the full-resolution level only, as a lower bound of the work done
        alg = 216.0 * W * H * D
        res["roofline"] = {"bound": "hbm", "kernel": "whole mgm_multi tile (pyramid of mgm calls)", "achieved": alg / (ms / (B * steps) * 1e-3) / 1e9,
                           "peak": ctx["peak"], "unit": "GB/s", "frac": alg / (ms / (B * steps) * 1e-3) / 1e9 / ctx["peak"], "traffic": None,
                           "note": "216 B x H x W x D of the full-resolution level / time of the whole tile"}
    del d_ref, d_sec, d_out, keep
    torch.cuda.empty_cache()
    return res, pairs


def extra_c3(ctx):
    """BASELINE configs[2]: 4096x4096 ROI, tile_size 512 (+ margins: 768x532), matcher mgm_multi, disp_range 256."""
    W, H, dmin, dmax = 768, 532, -128, 127
    res, pairs = _matcher_config(ctx, "mgm_multi", W, H, dmin, dmax, B=8, steps=2, nslots=4,
                                 label="BASELINE configs[2]: mgm_multi (-S 6, SUBPIX=2, REMOVESMALLCC=25, TSGM=4) on 768x532 tiles, 256 labels")
    if ctx["cpu"]:
        from oracle import oracle as O
        if O.have_ref():
            procs = max(1, (os.cpu_count() or 4) // 4)
            tiles = [(pairs[k % len(pairs)][0][:128], pairs[k % len(pairs)][1][:128]) for k in range(procs)]
            v, dt = _cpu_sample("mgm_multi", tiles, dmin, dmax, O.mgm_multi_params(), procs)
            res["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": procs, "kind": "reference",
                                   "sample": "%d strips of 768x128 px, 256 labels, one single-thread reference `mgm_multi` each, %.1f s wall" % (procs, dt)}
    return res


def extra_nodata(ctx):
    """configs[1] with 5 % no-data strips in both images: what a real rectified tile looks like."""
    a = ctx["a"]
    res, _ = _matcher_config(ctx, "mgm", a.size, a.size, a.dmin, a.dmax, B=8, steps=3, nslots=min(a.slots, 6), nan_border=0.05,
                             label="configs[1] with 5 % no-data strips in both images (DCT round trip of the matched image active, "
                                   "no-data sentinel range in the right view)")
    return res


def extra_c4(ctx):
    """BASELINE configs[3] as STRONG scaling: a fixed queue of 256 tiles 1026x1026, disp_range 192, pulled dynamically by the
    ranks from one shared counter (s2p_b200.tiles.DynamicQueue), host buffers in, host buffers out."""
    torch, eng, a = ctx["torch"], ctx["eng"], ctx["a"]
    from s2p_b200.engine import default_params
    from s2p_b200.synth import make_pair
    from s2p_b200.tiles import DynamicQueue
    W = H = 1026
    dmin, dmax, NT, CH = -96, 95, 256, 8
    D = dmax - dmin + 1
    p = default_params("mgm")
    base = [make_pair(H, W, dmin, dmax, seed=7000 + k)[:2] for k in range(8)]       # same on every rank
    keep = []
    # tile t = base tile t % 8 rolled by 31 (t // 8) rows: 256 distinct inputs, resident in page-locked host memory
    refs = [_pin(torch, keep, np.roll(base[t % 8][0], 31 * (t // 8), axis=0)) for t in range(NT)]
    secs = [_pin(torch, keep, np.roll(base[t % 8][1], 31 * (t // 8), axis=0)) for t in range(NT)]
    outs = ([_pin(torch, keep, np.empty((H, W), np.float32)) for _ in range(CH)], [_pin(torch, keep, np.empty((H, W), np.float32)) for _ in range(CH)],
            [_pin(torch, keep, np.empty((H, W), np.uint8)) for _ in range(CH)])
    nslots = min(6, a.slots)
    ok = 1.0
    try:
        eng.reserve(nslots, W, H, D)
        eng.mgm_batch(refs[:CH], secs[:CH], dmin, dmax, p, out=outs)               # warm-up (allocations, DCT tables)
    except Exception as e:
        ok, err = 0.0, e
    if ctx["world"] > 1:          # every rank enters the timed loops or none does
        tv = torch.tensor([ok], device=ctx["dev"])
        ctx["dist"].all_reduce(tv, op=ctx["dist"].ReduceOp.MIN)
        if tv.item() < 0.5:
            raise RuntimeError("set-up failed on a rank")
    elif not ok:
        raise err
    reps, took, walls = 2, 0, []
    for rep in range(reps):
        q = DynamicQueue(NT, CH, ctx["world"], key="s2pb_c4_rep%d" % rep)
        ctx["barrier"]()
        t0 = time.perf_counter()
        mine = 0
        while True:
            ids = q.next()
            if not ids:
                break
            eng.mgm_batch([refs[i] for i in ids], [secs[i] for i in ids], dmin, dmax, p,
                          out=tuple(o[:len(ids)] for o in outs))
            mine += len(ids)
        ctx["barrier"]()
        walls.append(ctx["max_over_ranks"](time.perf_counter() - t0))
        took = mine
    wall = min(walls)
    value = NT * W * H / wall / 1e6
    res = {"workload": "BASELINE configs[3] as a fixed queue: 256 tiles 1026x1026, 192 labels, algo mgm, pulled dynamically in chunks of 8 "
                       "from one shared counter by the ranks (no data-path collective)", "tile": [W, H], "labels": D, "tiles_total": NT,
           "metric": "disparity Mpix/s", "value": value, "unit": UNIT, "scaling": "strong", "seconds": wall, "gvoxel_per_s": value * D / 1e3,
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": NT * 2 * W * H * 4, "d2h_bytes_per_step": NT * (2 * W * H * 4 + W * H)},
           "tiles_taken_by_rank0": took, "tiles_in_flight": nslots,
           "note": "value == e2e: this configuration only exists with host buffers; best of %d passes over the queue" % reps}
    agg = []
    d = [torch.from_numpy(x).to(ctx["dev"]) for x in (base[0][0], base[0][1])]
    o = (torch.empty((H, W), dtype=torch.float32, device=ctx["dev"]), torch.empty((H, W), dtype=torch.float32, device=ctx["dev"]))
    for _ in range(3):
        eng.mgm_device(0, d[0].data_ptr(), d[1].data_ptr(), W, H, dmin, dmax, p, o[0].data_ptr(), o[1].data_ptr(), 0, 0, nodata_hint=0)
        eng.sync()
        agg.append(eng.last_timings(0))
    am = float(np.mean([x["aggregate"] for x in agg[1:]]))
    alg = 192.0 * W * H * D
    res["roofline"] = {"bound": "hbm", "kernel": "aggregate_kernel", "achieved": alg / (am * 1e-3) / 1e9, "peak": ctx["peak"], "unit": "GB/s",
                       "frac": alg / (am * 1e-3) / 1e9 / ctx["peak"], "kernel_ms": am, "algorithmic_bytes_per_launch": alg, "traffic": None,
                       "stage_ms": agg[-1]}
    if ctx["cpu"]:
        from oracle import oracle as O
        if O.have_ref():
            procs = max(1, (os.cpu_count() or 4) // 4)
            tiles = [(base[k % 8][0][:24], base[k % 8][1][:24]) for k in range(procs)]
            v, dt = _cpu_sample("mgm", tiles, dmin, dmax, O.mgm_params(), procs)
            res["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": procs, "kind": "reference",
                                   "sample": "%d strips of 1026x24 px, 192 labels, one single-thread reference `mgm` each, %.1f s wall" % (procs, dt)}
    del keep, refs, secs, outs
    return res


def extra_c5(ctx):
    """BASELINE configs[4]: tri-stereo -- two pairs per tile through the matcher, then the pixelwise merge of
    s2p.fusion.merge_n (s2p/fusion.py:25-68; here on the two disparity rasters, offsets = their means)."""
    torch, eng, a = ctx["torch"], ctx["eng"], ctx["a"]
    from s2p_b200.engine import default_params
    from s2p_b200.synth import make_pair
    W = H = 1024
    dmin, dmax, B, steps = -64, 63, 4, 2
    p = default_params("mgm")
    eng.reserve(min(a.slots, 8), W, H, dmax - dmin + 1)
    keep = []
    refs, secs = [], []
    for t in range(B):
        r, s2 = make_pair(H, W, dmin, dmax, seed=9000 + ctx["rank"] * B + t)[:2]
        refs += [_pin(torch, keep, r)] * 2
        secs += [_pin(torch, keep, s2), _pin(torch, keep, np.roll(s2, 3, axis=1))]     # third view: the second shifted by 3 px
    outs = ([_pin(torch, keep, np.empty((H, W), np.float32)) for _ in refs], [_pin(torch, keep, np.empty((H, W), np.float32)) for _ in refs],
            [_pin(torch, keep, np.empty((H, W), np.uint8)) for _ in refs])

    def step():
        eng.mgm_batch(refs, secs, dmin, dmax, p, out=outs)
        t0 = time.perf_counter()
        for t in range(B):
            eng.merge_n([outs[0][2 * t], outs[0][2 * t + 1]], [0.0, 3.0], "average_if_close", 1.0)
        return time.perf_counter() - t0
    step()
    ctx["barrier"]()
    t0 = time.perf_counter()
    fus = sum(step() for _ in range(steps))
    ctx["barrier"]()
    wall = ctx["max_over_ranks"](time.perf_counter() - t0)
    value = ctx["world"] * B * W * H * steps / wall / 1e6
    fus_ms = 1e3 * fus / (B * steps)
    res = {"workload": "BASELINE configs[4]: tri-stereo, per tile 2 pairs through algo mgm (1024x1024, 128 labels) + fusion.merge_n "
                       "(average_if_close) of the two rasters", "tile": [W, H], "labels": dmax - dmin + 1, "pairs_per_tile": 2,
           "metric": "fused-tile Mpix/s", "value": value, "unit": UNIT, "scaling": "weak",
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": B * (4 * W * H * 4 + 2 * W * H * 4), "d2h_bytes_per_step": B * (2 * (2 * W * H * 4 + W * H) + W * H * 4)},
           "fusion_ms_per_tile": fus_ms,
           "roofline": {"bound": "hbm", "kernel": "fusion_kernel (host-buffer call: H2D + kernel + D2H)", "achieved": 12.0 * W * H / (fus_ms * 1e-3) / 1e9,
                        "peak": ctx["peak"], "unit": "GB/s", "frac": 12.0 * W * H / (fus_ms * 1e-3) / 1e9 / ctx["peak"], "traffic": None,
                        "note": "12 B per pixel (two float32 in, one out) / wall time of s2pb_merge_n with pageable host buffers: PCIe-bound, not HBM-bound"},
           "note": "value == e2e (host buffers only)"}
    if ctx["cpu"]:
        import warnings
        from oracle import fusion_oracle as F
        t0 = time.perf_counter()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            F.merge_ref([outs[0][0][:64], outs[0][1][:64]], [0.0, 3.0], 1.0) if F.reference_average_if_close() else F.merge_port([outs[0][0][:64], outs[0][1][:64]], [0.0, 3.0])
        dt = time.perf_counter() - t0
        res["cpu_baseline"] = {"value": 64 * W / dt / 1e6, "unit": "Mpix/s (fusion only)", "cores": 1, "kind": "reference" if F.reference_average_if_close() else "port",
                               "sample": "merge of two 1024x64 strips through np.apply_along_axis(average_if_close), %.2f s" % dt}
    return res


def extra_warp(ctx):
    """The rectification warp of rectify_pair (3rdparty/homography): 1500x1500 source -> 1024x1024, a 12 degree rotation."""
    eng = ctx["eng"]
    rng = np.random.default_rng(5)
    sw = sh = 1500
    W = H = 1024
    src = (rng.integers(0, 4096, (sh, sw)).astype(np.float32))
    from s2p_b200.synth import _blur
    src = _blur(src.astype(np.float64)).astype(np.float32)
    th = np.deg2rad(12.0)
    c, s_ = np.cos(th), np.sin(th)
    R = np.array([[c, -s_, 0], [s_, c, 0], [0, 0, 1.0]])
    T = lambda x, y: np.array([[1, 0, x], [0, 1, y], [0, 0, 1.0]])
    Hm = T(W / 2, H / 2) @ R @ T(-sw / 2, -sh / 2)
    keep = []
    src = _pin(ctx["torch"], keep, src)                       # page-locked source and destination: the library DMAs from / to them
    dst = _pin(ctx["torch"], keep, np.empty((H, W), np.float32))
    for _ in range(3):
        out = eng.homography(src, Hm, W, H, out=dst)
    n = 20
    ctx["barrier"]()
    t0 = time.perf_counter()
    for _ in range(n):
        out = eng.homography(src, Hm, W, H, out=dst)
    ctx["barrier"]()
    wall = ctx["max_over_ranks"](time.perf_counter() - t0)
    value = ctx["world"] * n * W * H / wall / 1e6
    alg = 4.0 * sw * sh + 4.0 * W * H + 16.0 * sw * sh
    res = {"workload": "rectification warp: 1500x1500 float32 source -> 1024x1024, rotation 12 degrees (quintic B-spline, 2 x 2-pole prefilter)",
           "metric": "warped Mpix/s (output pixels)", "value": value, "unit": UNIT, "ms_per_warp": 1e3 * wall / n, "scaling": "weak",
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": sw * sh * 4, "d2h_bytes_per_step": W * H * 4},
           "roofline": {"bound": "hbm", "kernel": "prefilter + interpolation (whole host-buffer call)", "achieved": alg / (wall / n) / 1e9, "peak": ctx["peak"],
                        "unit": "GB/s", "frac": alg / (wall / n) / 1e9 / ctx["peak"], "traffic": None,
                        "note": "4 src + 4 dst + 16 src bytes per call (SURVEY.md 8d) / wall time of the host-buffer call (copies included)"},
           "valid_fraction": float(np.isfinite(out).mean()), "note": "value == e2e (the stand-alone warp is only exposed with host buffers, page-locked here; s2pb_rectify_match keeps the warped pair on the device)"}
    if ctx["cpu"]:
        from oracle import oracle as O
        if O.have_ref_homography():
            t0 = time.perf_counter()
            O.run_ref_homography(src, Hm, W, H)
            dt = time.perf_counter() - t0
            res["cpu_baseline"] = {"value": W * H / dt / 1e6, "unit": UNIT, "cores": 1, "kind": "reference",
                                   "sample": "one run of the reference resampler (oracle/_ref/homography_ref), PFM I/O included, %.2f s" % dt}
    return res


MULTI_RANK_EXTRA = ("C4_tile_queue_1026x1026x192_strong",)
EXTRA = [("C2_nodata_5pct", extra_nodata), ("C3_mgm_multi_256", extra_c3), ("C4_tile_queue_1026x1026x192_strong", extra_c4),
         ("C5_tristereo_fusion", extra_c5), ("rectification_warp", extra_warp)]


def main():
    a = parse()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if a.impl == "reference":
        run_reference(a, rank, world)
    else:
        run_ours(a, rank, world, local_rank)


if __name__ == "__main__":
    main()
