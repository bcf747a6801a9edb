#!/usr/bin/env python
"""bench.py — frames/sec of the splat hot path (sort + project + bin + raster) on B200.

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle restatement)
    python bench.py ... --dump-outputs DIR                   # also save the frame of the last timed step (frame_outputs)

A "step" is one full frame of the workload: the worker sort request plus the instanced draw
(reference index.js:438-455 + 184-207), synchronously with the same camera.
N = 1 workload = BASELINE.json configs[1]: train-like 1 M synthetic splats, 1920x1080, fixed camera; the same run
then also times configs[2] (6 M, orbit) and configs[3] (20 M, 3840x2160, cutout) and prints them under
`other_configs`.  N > 1 (see parallel_mode): by default every rank renders every N-th frame of the stream from its own
replica of the scene (weak scaling, no data-path collective); `--parallel tiles` (default for the 80 M scene) shards ONE
frame by screen bin columns over the ranks and exchanges the finished tiles (strong scaling).

`value`  : frames/s with the scene resident in HBM and the frame left in HBM (device-timed: one CUDA-event pair around
           the K steps on the library's stream, three frames in flight, L2 flushed between steps inside the region).
`e2e`    : frames/s through gs_render_async/gs_wait with HOST buffers: camera matrices in, RGBA8 frame out to pinned
           host memory, both copies inside the timed region.
`parity` : the timed configuration's GPU frame against the CPU oracle's frame of the same inputs (max abs error on
           float RGBA, LSB histogram on RGBA8, exactness of the sort) — the run exits non-zero above 1e-3.
"""
from __future__ import annotations

import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "frames/sec @1920x1080 (sort + splat raster, 1 M synthetic train-like splats)"
METRICS = {
    "train_1m_1080p": METRIC,
    "bicycle_6m_1080p_orbit": "frames/sec @1920x1080 (sort + splat raster, 6 M synthetic splats, 360-degree orbit, re-sort per frame)",
    "synth_20m_2160p_cutout": "frames/sec @3840x2160 (sort + splat raster, 20 M synthetic splats, cutout box)",
    "synth_80m_1080p": "frames/sec @1920x1080 (sort + splat raster, 80 M synthetic splats)",
}
FRAME_TOL = 1e-3
DTYPE = "f64 sort keys + f32 shading"
DUMP_BYTES = 64_000_000  # --dump-outputs: total size of the .npy files


def load_gsplat(gs):
    """The CUDA library as build() left it in the tree.  One that is missing or older than its sources is compiled into
    a temporary directory instead: the bench writes nothing into the tree, which may be read-only."""
    if not gs.build.stale():
        return gs._lib.load()
    with tempfile.TemporaryDirectory(prefix="gsplat_bench_") as tmp:
        return gs._lib.load(gs.build.build_library(out=os.path.join(tmp, "libgsplat_b200.so")))


def load_oracle():
    """The CPU oracle, found or compiled like the CUDA library in load_gsplat()."""
    from oracle import oracle as orc
    if orc.stale():
        with tempfile.TemporaryDirectory(prefix="gsplat_bench_") as tmp:
            orc.lib(orc.build(out=os.path.join(tmp, "libgs_oracle.so")))
    return orc


def frame_outputs(frame: np.ndarray) -> dict:
    """--dump-outputs arrays of one (H, W, 4) RGBA8 frame (row 0 = bottom), as float32 byte values: `frame` when the
    whole frame fits DUMP_BYTES, otherwise a fixed seeded sample of its pixels, `frame_pixels` (k, 4), and their
    row-major pixel indices, `frame_pixel_index` (k,) float64.  Same frame -> same arrays."""
    f = np.ascontiguousarray(frame, np.float32)
    if f.nbytes <= DUMP_BYTES - 4096:  # room for the .npy headers
        return {"frame": f}
    px = f.reshape(-1, f.shape[-1])
    k = (DUMP_BYTES - 4096) // (px.itemsize * px.shape[1] + 8)
    idx = np.sort(np.random.default_rng(0).choice(px.shape[0], k, replace=False))
    return {"frame_pixels": px[idx], "frame_pixel_index": idx.astype(np.float64)}


def write_outputs(out_dir: str, arrays: dict) -> None:
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def algorithmic_bytes(st: dict) -> dict:
    """SURVEY.md 8(d) per-frame algorithmic bytes, from the counters the library returns."""
    # D = 16x16 tile instances whose tile really meets the r<=2 footprint (SURVEY.md 8: "D = sum of 16x16 tiles touched"),
    # counted exactly by a GS_RENDER_STATS frame.  The library itself bins to 96x96-pixel bins (~5x fewer instances) and
    # culls per tile inside the raster, so it MOVES fewer bytes than this formula charges.
    N, V, V2, D, T = st["n_splats"], st["n_sorted"], st["n_visible"], st["n_tile_instances"], st["n_tiles"]
    P = st["width"] * st["height"]
    if st.get("n_slabs"):
        # front-to-back slab path (DESIGN.md 5.1): the one-pass formula would charge work this path never does (bins that
        # closed), so the bytes are those of the passes it really needs.  R slabs ran over E draw-order entries, K bin
        # instances were kept.
        R, E, K = st["n_slabs_run"], st["n_slab_entries"], st["n_instances_kept"]
        a = 20 * N + 8 * N + 4 * N + 4 * N    # cull read, fp32 depth out and back in (range first, then key), key write, offsets pass
        b = R * 4 * N + E * (6 + 24 + 24 + 32) + 80 * K + 8 * T * R  # per slab: key scan; per entry: compact, 2 radix passes, project
        r = 36 * K + 32 * P + 4 * P           # records + pixel state once + the frame
        return {"sort": a, "project": 0, "bin": b, "raster": r, "total": a + b + r}
    return {
        "sort": 20 * N + 8 * V,               # K1: 16 B centre + 4 B sizeAlpha read, depth + index write
        "project": 8 * V + 16 * V + 32 * V2,  # K2 (without the key emission, counted under bin)
        "bin": 8 * D + 68 * D + 4 * D + 8 * T,  # key emission + K3 4 passes + K4
        "raster": 36 * D + 4 * P,             # K5: sorted values + 32 B record per instance + RGBA8 frame
        "total": 20 * N + 32 * V + 32 * V2 + 116 * D + 8 * T + 4 * P,
    }


def parallel_mode(args) -> str:
    """How N > 1 GPUs are used.  `frames`: every rank holds the whole scene and renders every N-th frame of the stream
    (independent units, no data-path collective, weak scaling: the north star shards the splats "only when the scene
    outgrows one GPU").  `tiles`: ONE frame is sharded by screen bin columns over the ranks and the finished tiles are
    exchanged (strong scaling; the default for the 80 M-splat configuration)."""
    if args.parallel != "auto":
        return args.parallel
    return "tiles" if args.workload == "synth_80m_1080p" else "frames"


def parallelism_label(world: int, exchange: str, mode: str = "tiles") -> str:
    if world == 1:
        return "1 GPU"
    if mode == "frames":
        return f"frame-parallel x{world}: every rank renders every {world}-th frame of the stream from its own replica of the splat table, no data-path collective"
    if exchange == "p2p":
        return f"screen-tile-column sharding x{world}, raster fused with the exchange over NVLink peer memory"
    return f"screen-tile-column sharding x{world} + NCCL all-gather of RGBA8 tiles"


def config_block(args, workload: str, n: int, w: int, h: int, orbit: bool) -> dict:
    """The `config` object: IDENTICAL in both arms for the same command line (the driver compares them)."""
    return {"workload": workload, "n_splats": n, "width": w, "height": h, "camera": "orbit-120" if orbit else "fixed",
            "parallelism": parallelism_label(args.gpus, args.exchange, parallel_mode(args)),
            "l2": "GPU arm: flushed between timed steps (160 MiB memset on the raster stream, INSIDE the timed region)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,utilization.gpu,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, uuid: str):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", uuid, f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self) -> dict:
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, smax, power, reasons = [], [], [], set()
        for r in rows:
            if len(r) < 9:
                continue
            try:
                util = float(r[3])
                if util >= 10.0:  # under load
                    sm.append(float(r[0]))
                smax.append(float(r[1]))
                power.append(float(r[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(rows), "samples_under_load": len(sm),
                "reasons": sorted(reasons)}


def build_scene(gs, workload: str, splats: int = 0):
    """rows + the frame list of a workload (one frame, or the 120 orbit steps of config 3)."""
    sc = gs.scenes
    n, w, h, seed, cutout = sc.CONFIGS[workload]
    if splats:
        n = splats
    rows = gs.synth_splats(n, seed)
    if "orbit" in workload:  # config 3: 120-step 360 degree yaw orbit, re-sorted every frame
        frames = [sc.make_frame(sc.orbit_camera(w, h, i), sc.demo_object(), w, h) for i in range(120)]
    else:
        frames = [sc.make_frame(sc.fixed_camera(w, h), sc.demo_object(), w, h, sc.demo_cutout() if cutout else None)]
    return rows, frames, n, w, h


# ------------------------------------------------------------------------------------------------------
# the reference's own CPU implementation of the path (oracle restatement; Node/WebGL are absent from the image)
# ------------------------------------------------------------------------------------------------------
def cpu_threads(orc):
    """Raster workers = one per PHYSICAL core of this process's affinity mask, each pinned (round 1's unpinned
    one-thread-per-logical-CPU run swung 4x between two hosts)."""
    cpus = orc.physical_cpus()
    orc.set_affinity(cpus)
    return len(cpus)


def cpu_pick_band(orc, cs, cc, order, fr, w, h, budget_s: float, threads: int):
    """Rows to shade per step so that one raster pass fits the budget (full frame when it does)."""
    band = max(16, h // 16)
    y0 = (h - band) // 2
    t0 = time.perf_counter()
    orc.render(cs, cc, order, fr.proj, fr.modelview, w, h, fr.focal, nthreads=threads, rows=(y0, y0 + band))
    est_full = (time.perf_counter() - t0) * h / band
    if est_full <= budget_s:
        return (0, h)
    nb = int(max(band, min(h, h * budget_s / est_full)))
    return ((h - nb) // 2, (h - nb) // 2 + nb)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    gs = importlib.import_module("aframe-gaussian-splatting_b200")
    orc = load_oracle()
    rows, frames, n, w, h = build_scene(gs, args.workload, args.splats)
    threads = cpu_threads(orc)
    cs, cc, m = orc.pack(rows)
    per_step = 150.0 / max(1, args.steps + args.warmup)
    order = orc.sort(m, frames[0].view, frames[0].cutout)
    band = cpu_pick_band(orc, cs, cc, order, frames[0], w, h, per_step, threads)
    t_sort, t_rast = [], []
    for i in range(args.warmup + args.steps):
        fr = frames[i % len(frames)]
        t0 = time.perf_counter()
        order = orc.sort(m, fr.view, fr.cutout)   # ONE thread: the reference has one Web Worker (index.js:229)
        t1 = time.perf_counter()
        orc.render(cs, cc, order, fr.proj, fr.modelview, w, h, fr.focal, nthreads=threads, rows=band)
        t2 = time.perf_counter()
        if i >= args.warmup:
            t_sort.append(t1 - t0)
            t_rast.append((t2 - t1) * h / (band[1] - band[0]))
    step = np.asarray(t_sort) + np.asarray(t_rast)
    ms = 1000.0 * float(np.median(step))  # median step: robust against a noisy host
    fps = 1000.0 / ms
    sample = (f"sortSplats restatement on 1 thread + software raster on {threads} pinned threads (one per physical core); "
              + ("full frames" if band == (0, h) else f"rows {band[0]}..{band[1]} of {h} shaded per step, raster time scaled by {h}/{band[1]-band[0]}")
              + "; value = 1 / median step")
    line = {"impl": "reference", "metric": METRICS.get(args.workload, METRIC), "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak" if (args.gpus > 1 and parallel_mode(args) == "frames") else "strong",
            "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
            "config": config_block(args, args.workload, n, w, h, len(frames) > 1),
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port", "sample": sample,
                             "nproc": os.cpu_count(), "sort_ms_median": 1000 * float(np.median(t_sort)),
                             "raster_ms_median": 1000 * float(np.median(t_rast)), "ms_per_step_mean": 1000 * float(np.mean(step)),
                             "ms_per_step_min": 1000 * float(np.min(step)), "ms_per_step_max": 1000 * float(np.max(step))},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------
def parity_block(gs, orc, ctx, rows, fr, w, h, threads):
    """GPU frame vs oracle frame of the same inputs, at the size being timed.  Also returns the CPU timings of the oracle
    calls (the cpu_baseline leg: the oracle is executed here only as checker / baseline, never on the product path)."""
    t0 = time.perf_counter()
    cs, cc, m = orc.pack(rows)
    t_pack = time.perf_counter() - t0
    ts = []
    for _ in range(3):
        t0 = time.perf_counter()
        order = orc.sort(m, fr.view, fr.cutout)
        ts.append(time.perf_counter() - t0)
    t0 = time.perf_counter()
    exp, est = orc.render(cs, cc, order, fr.proj, fr.modelview, w, h, fr.focal, nthreads=threads)
    t_render = time.perf_counter() - t0
    got_order = ctx.sort(fr.view, fr.cutout)
    sort_exact = bool(np.array_equal(got_order, order))
    got = ctx.render(fr, fmt=gs.GS_FORMAT_RGBA32F)
    err = np.abs(got - exp)
    max_err = float(err.max())
    where = [int(x) for x in np.unravel_index(int(err.argmax()), err.shape)]
    got8 = ctx.render(fr, fmt=gs.GS_FORMAT_RGBA8)
    e8 = np.floor(np.clip(exp, 0, 1) * 255.0 + 0.5).astype(np.int32)
    d8 = np.abs(got8.astype(np.int32) - e8)
    tot = float(d8.size)
    hist = {"0": float((d8 == 0).sum() / tot), "1": float((d8 == 1).sum() / tot), "2": float((d8 == 2).sum() / tot),
            ">2": float((d8 > 2).sum() / tot)}
    cov = orc.coverage_check(cs, cc, order, fr.proj, fr.modelview, w, h, fr.focal, nthreads=threads)
    par = {"oracle": "oracle/gs_oracle.c (CPU restatement of index.js; parity unpinned: the reference holds no vectors)",
           "frame": f"{w}x{h}, full frame, all {len(order)} sorted splats", "tolerance": FRAME_TOL,
           "max_abs_err": max_err, "argmax_yxc": where, "mean_abs_err": float(err.mean()),
           "lsb_hist": hist, "sort_exact": sort_exact, "n_sorted": int(len(order)), "oracle_fragments": int(est["fragments"]),
           "ok": bool(sort_exact and max_err <= FRAME_TOL and hist[">2"] == 0.0),
           "gl_coverage_check": dict(cov, note="affine vPosition (both rasters) vs GL barycentric interpolation of the quad's two "
                                                "triangles in fp64 (independent of a1/a2): pairs whose keep/discard decision differs")}
    t_sort = float(np.median(ts))
    cpu = {"value": 1.0 / (t_sort + t_render), "unit": "frames/s", "cores": threads, "kind": "port", "nproc": os.cpu_count(),
           "sort_ms_1thread": 1000 * t_sort, "raster_ms": 1000 * t_render, "pack_ms_1thread": 1000 * t_pack,
           "sample": f"one full frame: sortSplats restatement on 1 thread (median of 3) + software raster on {threads} pinned threads"}
    return par, cpu


def run_ours(args):
    import torch
    import torch.distributed as dist
    gs = importlib.import_module("aframe-gaussian-splatting_b200")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU path")
    # scenes first: the generator forks worker processes, which must happen before this process owns a CUDA context
    names = [args.workload]
    if world == 1 and args.workload == "train_1m_1080p" and not args.no_other_configs and not args.splats:
        names += ["bicycle_6m_1080p_orbit", "synth_20m_2160p_cutout"]
    scenes = {}
    for nm in names:
        t0 = time.perf_counter()
        scenes[nm] = build_scene(gs, nm, args.splats if nm == args.workload else 0)
        if rank == 0:
            sys.stderr.write(f"[bench] scene {nm}: {scenes[nm][2]} splats generated in {time.perf_counter() - t0:.1f} s\n")

    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ.pop("NCCL_DEBUG")  # its banner goes to stdout; keep stdout to the one JSON line
        # the all-gather of finished tiles is latency-critical and tiny: give NCCL's stream the same (highest) priority
        # as the library's sort/bin streams, otherwise its kernels queue behind them on every rank and the ranks skew
        opts = None
        try:
            opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
        except Exception:
            pass
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local), pg_options=opts)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    load_gsplat(gs)
    ctx = gs.SplatContext(local)
    stream = torch.cuda.ExternalStream(ctx._lib.gs_stream(ctx._h), device=dev)
    with torch.cuda.stream(stream):
        flush = torch.empty(160 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    stream.synchronize()
    os.environ.setdefault("GS_BENCH", "1")
    uuid = str(torch.cuda.get_device_properties(dev).uuid)
    uuid = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
    peak, peak_src = load_peaks()
    dump = {}  # --dump-outputs arrays of the headline configuration

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x: float) -> float:
        if world == 1:
            return float(x)
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def measure(name: str, steps: int, headline: bool, mode: str = None) -> dict:
        mode = mode or parallel_mode(args)
        sharded = world > 1 and mode == "tiles"   # one frame split over the ranks
        afr = world > 1 and mode == "frames"      # whole frames dealt round-robin to the ranks
        rows, frames, n, w, h = scenes[name]
        orbit = len(frames) > 1
        fr = frames[0]
        # ---- load: progressive push in 4 M-row chunks (index.js:259-298), timed on the host clock ----
        ctx.clear()
        ctx.set_shard(rank if sharded else 0, world if sharded else 1)
        chunk = 4 << 20
        ctx.reserve(n)                      # initGL(numVertexes): size the table once (index.js:248-251)
        ctx.push_splats(rows[:min(n, 1 << 18)])  # first touch of the staging buffers is not part of the rate
        ctx.read_packed(0, 1)               # (waits for the push stream)
        ctx.clear()
        t0 = time.perf_counter()
        for first in range(0, n, chunk):
            ctx.push_splats(rows[first:first + chunk])
        ctx.read_packed(0, 1)
        t_push = time.perf_counter() - t0
        tiles_per_rank = max(ctx.owned_tiles(w, h, r, world) for r in range(world))
        flags = gs.GS_RENDER_OUT_DEVICE | (gs.GS_RENDER_OUT_TILED if sharded else 0)
        p_dev = [ctx.make_params(f, fmt=gs.GS_FORMAT_RGBA8, flags=flags) for f in frames]
        p_host = [ctx.make_params(f, fmt=gs.GS_FORMAT_RGBA8, flags=0) for f in frames]
        nf = len(frames)
        with torch.cuda.stream(stream):
            frames_dev = [torch.zeros(h * w * 4, dtype=torch.uint8, device=dev) for _ in range(4)]
            tiles_bufs = [torch.zeros(tiles_per_rank * 1024, dtype=torch.uint8, device=dev) for _ in range(3)] if sharded else None
            gath_bufs = [torch.zeros(world * tiles_per_rank * 1024, dtype=torch.uint8, device=dev) for _ in range(3)] if sharded else None
        stream.synchronize()

        # ---- multi-GPU exchange: fused raster + peer stores over NVLink (default) or NCCL all-gather of tiles ----
        use_peer = sharded and args.exchange == "p2p"
        if use_peer:
            ok = 1
            try:  # every rank must take the same path: agree on whether the peer mapping worked everywhere
                handles = [None] * world
                dist.all_gather_object(handles, ctx.peer_export(h * w * 4))
                ctx.peer_import(rank, world, handles)
            except Exception as e:  # no peer access / IPC on this box
                sys.stderr.write(f"[rank {rank}] fused exchange unavailable ({e}); falling back to the NCCL all-gather\n")
                ok = 0
            flag = torch.tensor([ok], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            use_peer = bool(flag.item())
        if use_peer:
            ctx.render_raw(ctx.make_params(fr, fmt=gs.GS_FORMAT_RGBA8, flags=gs.GS_RENDER_OUT_DEVICE), frames_dev[0].data_ptr())  # sizes the instance buffers
            dist.barrier()
            peer_dev = ctx.make_params(fr, fmt=gs.GS_FORMAT_RGBA8, flags=gs.GS_RENDER_OUT_DEVICE | gs.GS_RENDER_OUT_PEER)
            peer_host = ctx.make_params(fr, fmt=gs.GS_FORMAT_RGBA8, flags=gs.GS_RENDER_OUT_PEER)

        def fidx(i):
            """frame of the stream this rank renders at its step i (frame-parallel: rank r takes frames r, r+N, ...)"""
            return (gs.dist.rank_frame(i, rank, world) if afr else i) % nf

        def submit_device(i):
            """enqueue frame i on the library's streams (no host synchronisation); returns its ticket"""
            if use_peer:
                return ctx.render_async(peer_dev, 1)  # the assembled frame lands in the shared ring
            if not sharded:
                return ctx.render_async(p_dev[fidx(i)], frames_dev[i % 4].data_ptr())
            t = ctx.render_async(p_dev[i % nf], tiles_bufs[i % 3].data_ptr())
            with torch.cuda.stream(stream):
                dist.all_gather_into_tensor(gath_bufs[i % 3], tiles_bufs[i % 3])
            ctx.assemble_tiles(gath_bufs[i % 3].data_ptr(), tiles_per_rank, world, w, h, gs.GS_FORMAT_RGBA8, frames_dev[i % 3].data_ptr())
            return t

        def run_pipeline(submit, k, collect=None, depth=3, tickets=None):
            """k frames, at most `depth` outstanding (3: sort(i) | bin(i-1) | raster(i-2); 4 when frames also cross PCIe:
            + copy(i-3)); one CUDA-event pair on the library's stream brackets everything (the L2 flushes between steps
            included).  The frames' tickets are appended to `tickets` when a list is given."""
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            tickets = [] if tickets is None else tickets
            with torch.cuda.stream(stream):
                r0.record(stream)
            for i in range(k):
                with torch.cuda.stream(stream):
                    flush.zero_()  # L2 flush between timed iterations
                tickets.append(submit(i))
                if i >= depth - 1:
                    st = ctx.wait(tickets[i - (depth - 1)])
                    if collect is not None:
                        collect.append(st.as_dict())
            for t in tickets[max(0, len(tickets) - (depth - 1)):]:
                st = ctx.wait(t)
                if collect is not None:
                    collect.append(st.as_dict())
            with torch.cuda.stream(stream):
                r1.record(stream)
            stream.synchronize()
            return r0.elapsed_time(r1)

        run_pipeline(submit_device, max(args.warmup, 3))
        # ... and keep warming until the GPU has been busy for ~0.3 s: a freshly woken GPU (the second rank's in
        # particular) needs longer than three 0.3 ms frames to reach its clocks.  Same count on every rank.
        t_w = time.perf_counter()
        run_pipeline(submit_device, 50)
        per50 = allmax(time.perf_counter() - t_w)
        for _ in range(int(min(40, max(0.0, 0.3 - per50) / max(per50, 1e-4)))):
            run_pipeline(submit_device, 50)
        sampler = ClockSampler(uuid) if rank == 0 else None

        # ---- value: device-resident frames ----
        barrier()
        timed = []
        my_ms = run_pipeline(submit_device, steps, depth=3 if sharded else args.value_depth, tickets=timed)
        if headline and rank == 0 and args.dump_outputs:
            # the frame of the last timed step, read before the untimed frames below reuse its buffer
            last = np.empty((h, w, 4), np.uint8)
            src = ctx.peer_frame(timed[-1]) if use_peer else frames_dev[(steps - 1) % (3 if sharded else 4)].data_ptr()
            ctx.memcpy_d2h(last, src, last.nbytes)
            dump.update(frame_outputs(last))
        total_ms = allmax(my_ms)
        barrier()
        if world > 1:
            sys.stderr.write(f"[bench] rank {rank}: {my_ms / steps:.4f} ms per step (max over ranks {total_ms / steps:.4f})\n")
        units = world if afr else 1  # frames finished per step across the job
        ms_per_step = total_ms / steps
        fps = units * 1000.0 / ms_per_step

        # ---- un-overlapped frames (one in flight) for the per-stage / roofline numbers: with three frames in flight the
        #      stages of consecutive frames run concurrently and their individual durations stretch ----
        lat_stats = []
        for i in range(max(5, min(steps, 20))):
            with torch.cuda.stream(stream):
                flush.zero_()
            lat_stats.append(ctx.wait(submit_device(i)).as_dict())

        # ---- one diagnostic frame (untimed): exact D and the raster's pixel-splat pair counters ----
        p_stats = ctx.make_params(fr, fmt=gs.GS_FORMAT_RGBA8, flags=flags | gs.GS_RENDER_STATS)
        full_stats = ctx.wait(ctx.render_async(p_stats, (tiles_bufs[0] if sharded else frames_dev[0]).data_ptr())).as_dict()

        # ---- e2e: host buffers through the public C-ABI call, copies inside the timed region ----
        host_frames = [ctx.pinned_array((h, w, 4), np.uint8) for _ in range(4)]
        e2e_depth = 3 if sharded else 4  # the tile-sharded modes keep their three-entry exchange rings
        if not sharded:
            def submit_host(i):
                return ctx.render_async(p_host[fidx(i)], host_frames[i % 4].ctypes.data)
        elif use_peer:
            def submit_host(i):
                return ctx.render_async(peer_host, host_frames[i % 3].ctypes.data)
        else:
            def submit_host(i):
                t = submit_device(i)
                with torch.cuda.stream(stream):  # frame back to pinned host memory, stream-ordered after the un-tiling
                    torch.from_numpy(host_frames[i % 3].reshape(-1)).copy_(frames_dev[i % 3], non_blocking=True)
                return t
        run_pipeline(submit_host, 4, depth=e2e_depth)
        barrier()
        e2e_ms = allmax(run_pipeline(submit_host, steps, depth=e2e_depth)) / steps
        barrier()
        e2e = {"value": units * 1000.0 / e2e_ms, "unit": "frames/s", "ms_per_step": e2e_ms,
               "h2d_bytes_per_step": units * C.sizeof(gs.GsRenderParams), "d2h_bytes_per_step": units * h * w * 4,
               "frames_outstanding": e2e_depth,
               "note": "gs_render_async/gs_wait with host buffers, up to four tickets open (sort | bin | raster | copy): the camera matrices go in as one small "
                       "H2D copy, the RGBA8 frame comes back to pinned host memory on a copy stream while the next frame renders; "
                       "the timed region (one CUDA-event pair around all K steps) includes every copy and the L2 flushes"}

        # keep the GPU loaded long enough for nvidia-smi to observe the clocks under this workload.  The iteration count
        # is derived from the all-reduced step time, so every rank issues the same number of collectives.
        for _ in range(int(min(4000, max(10, (1200.0 if headline else 600.0) / max(ms_per_step, 1e-3))))):
            ctx.wait(submit_device(0))
        clocks = sampler.stop() if sampler is not None else None

        # ---- multi-GPU: the sharded frame must equal the frame one GPU renders alone ----
        frame_check = None
        if sharded:
            got = np.empty((h, w, 4), np.uint8)
            if use_peer:
                t = ctx.render_async(peer_dev, 1)
                ctx.wait(t)
                ctx.memcpy_d2h(got, ctx.peer_frame(t), got.nbytes)
            else:
                ctx.wait(submit_device(0))
                ctx.synchronize()
                got = frames_dev[0].cpu().numpy().reshape(h, w, 4).copy()
            barrier()
            if rank == 0:
                ctx.set_shard(0, 1)
                ref = ctx.render(fr, fmt=gs.GS_FORMAT_RGBA8)
                ctx.set_shard(rank, world)
                d = np.abs(got.astype(np.int32) - ref.astype(np.int32))
                frame_check = "bit-identical" if int(d.max()) == 0 else f"differs: max {int(d.max())} LSB on {int((d > 0).sum())} channel values"
            barrier()

        if afr:  # every rank renders the SAME reference frame: the pictures must agree bit for bit across the ranks
            ref = ctx.render(fr, fmt=gs.GS_FORMAT_RGBA8)
            hsh = int.from_bytes(__import__("hashlib").sha256(ref.tobytes()).digest()[:7], "little")
            t = torch.tensor([hsh], device=dev, dtype=torch.int64)
            lst = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(lst, t)
            same = all(int(x.item()) == hsh for x in lst)
            frame_check = "bit-identical" if same else "differs: the ranks' frames of the same camera have different hashes"

        res = None
        if rank == 0:
            st = {k: float(np.mean([s[k] for s in lat_stats])) for k in lat_stats[0]}
            for k in ("n_splats", "n_sorted", "n_visible", "n_instances", "n_instances_kept", "n_tiles", "width", "height", "kernel_launches", "n_dropped",
                      "n_slabs", "n_slabs_run", "n_slab_entries"):
                st[k] = int(lat_stats[0][k])
            for k2 in ("n_tile_instances", "n_records_streamed", "n_pair_tests", "n_pair_hits"):
                st[k2] = int(full_stats[k2])
            ab = algorithmic_bytes(st)
            stage_ms = {"sort": st["ms_sort"], "project": st["ms_project"], "bin": st["ms_bin"], "raster": st["ms_raster"]}
            dom = max(stage_ms, key=stage_ms.get)

            def roof(nm):
                ms = stage_ms[nm]
                ach = ab[nm] / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
                return {"bytes": ab[nm], "ms": ms, "achieved_gbs": ach, "frac": ach / peak}
            # DRAM traffic is a MEASUREMENT of one profiled launch (ncu --set full): quoted only for the exact configuration
            # profiles/traffic.json was captured on (N = 1, config 2), null everywhere else
            traffic = None
            tp = os.path.join(ROOT, "profiles", "traffic.json")
            if world == 1 and name == "train_1m_1080p" and not args.splats and os.path.exists(tp):
                try:
                    traffic = json.load(open(tp)).get(dom)
                except Exception:
                    traffic = None
            r = roof(dom)
            slab_info = None
            if st["n_slabs"]:
                slab_info = {"scheduled": st["n_slabs"], "run": st["n_slabs_run"], "entries": st["n_slab_entries"],
                             "note": "front-to-back slab path: stages are keys (sort) / slab loop without its rasters (bin) / rasters + resolve; "
                                     "bytes per stage are the slab path's own passes (bench.py algorithmic_bytes), not the one-pass formula"}
            kernels = {"sort": "k_depth_cull+k_radix_{hist,scan,scatter}<D1,D2>", "project": "k_project",
                       "bin": "k_count+k_emit_entries+k_radix_{hist,scan,scatter}<T1>(+<T2>+k_tile_ranges above 256 bins)", "raster": "k_raster"}
            res = {
                "metric": METRICS.get(name, METRIC), "value": fps, "unit": "frames/s", "ms_per_step": ms_per_step,
                "config": dict(config_block(args, name, n, w, h, orbit), parallelism=parallelism_label(world, args.exchange, mode)),
                "scaling": "weak" if afr else "strong",
                "counters": {k: st[k] for k in ("n_splats", "n_sorted", "n_visible", "n_instances", "n_instances_kept", "n_tile_instances", "n_tiles", "n_dropped")},
                "raster_pairs": {"tested": st["n_pair_tests"], "useful": st["n_pair_hits"],
                                 "useful_frac": st["n_pair_hits"] / max(1, st["n_pair_tests"]),
                                 "bin_records_streamed": st["n_records_streamed"], "tile_instances": st["n_tile_instances"],
                                 "note": "pixel-splat pairs evaluated by live pixels vs pairs blended (r^2 <= 4), from one GS_RENDER_STATS frame "
                                         "that walks every bin list to its end (a timed frame stops a tile once its pixels are saturated)"},
                "msplats_per_s": n * fps / 1e6,
                "e2e": e2e,
                "gpu_launches": (int(st["kernel_launches"]) + (2 if use_peer else (1 if sharded else 0))) * steps * units,
                "clocks": clocks,
                "roofline": {"kernel": kernels[dom], "bound": "hbm", "achieved": r["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": r["frac"],
                             "traffic": traffic, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": ab[dom], "ms_per_launch": stage_ms[dom],
                             "note": "k_raster is FP32-pipe bound (one exp + ~16 fp32 ops per covered pixel-splat pair), reported against HBM as SURVEY.md 8d prescribes"},
                "stages": {k: roof(k) for k in stage_ms},
                "frame": {"bytes": ab["total"], "ms_device": st["ms_total"], "achieved_gbs": ab["total"] / (st["ms_total"] * 1e-3) / 1e9,
                          "frac": ab["total"] / (st["ms_total"] * 1e-3) / 1e9 / peak},
                "push": {"msplats_per_s": n / t_push / 1e6, "n": n, "ms": 1000 * t_push,
                         "note": "gs_push_splats of raw 32 B rows from pageable host memory in 4 M-row chunks, device-side pack included"},
            }
            if slab_info:
                res["slabs"] = slab_info
                res["roofline"]["kernel"] = {"sort": "k_depth_cull+k_keys+k_slab_plan+k_compact_count_all+k_compact_scan_all",
                                             "bin": "per slab: k_compact_write+k_radix<S1,D2>+k_project<entries>+k_count+k_emit_entries+k_radix<T1>",
                                             "raster": "k_raster<slab> per slab + k_resolve", "project": "-"}[dom]
            if frame_check is not None:
                res["frame_check"] = frame_check
            if world == 1 and not args.no_cpu_baseline:
                orc = load_oracle()
                threads = cpu_threads(orc)
                par, cpu = parity_block(gs, orc, ctx, rows, frames[40 % nf], w, h, threads)
                res["parity"] = par
                res["cpu_baseline"] = cpu
        return res

    head = measure(args.workload, args.steps, True)
    alt = None
    if world > 1 and parallel_mode(args) == "tiles" and args.parallel == "auto":
        # the tile-sharded frame replicates the O(N) passes of the path on every rank; the same job dealt out as whole
        # frames (every rank holds the scene: 2.9 GB of 180 GB at 80 M splats) is printed beside it
        try:
            a = measure(args.workload, max(5, min(args.steps, 10)), False, mode="frames")
            if a is not None:
                alt = {k: a[k] for k in ("value", "unit", "ms_per_step", "scaling", "e2e", "frame_check", "clocks") if k in a}
                alt["parallelism"] = a["config"]["parallelism"]
        except Exception as e:
            alt = {"error": str(e)}
    others = []
    for nm in names[1:]:
        try:
            o = measure(nm, max(5, min(args.steps, 12)), False)
            if o is not None:
                o["steps"] = max(5, min(args.steps, 12))
                others.append(o)
        except Exception as e:  # a secondary configuration must not take the headline down
            others.append({"workload": nm, "error": str(e)})
    rc = 0
    if rank == 0:
        line = {"metric": head["metric"], "value": head["value"], "unit": "frames/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": head["ms_per_step"], "higher_is_better": True,
                "scaling": head["scaling"],
                "vs_baseline": None, "dtype": DTYPE, "data": "synthetic"}
        line.update({k: v for k, v in head.items() if k not in line})
        line["pipeline"] = ("three frames in flight: frame k is rasterised (low-priority stream) while frame k+1 is binned and frame "
                            "k+2 sorted/projected (high-priority streams); ms_per_step is the steady-state frame period, stages/roofline/frame "
                            "are from un-overlapped frames (one in flight) timed with the same CUDA events")
        if others:
            line["other_configs"] = others
        if alt is not None:
            line["alt_parallel"] = alt
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            write_outputs(args.dump_outputs, dump)
        bad = [x for x in [head] + others if isinstance(x.get("parity"), dict) and not x["parity"]["ok"]]
        if bad:
            sys.stderr.write("[bench] PARITY FAILURE: " + ", ".join(f"{x['config']['workload']} max_abs_err={x['parity']['max_abs_err']:.3g}" for x in bad) + "\n")
            rc = 1
        if head.get("frame_check") not in (None, "bit-identical"):
            sys.stderr.write(f"[bench] FRAME CHECK FAILURE: {head['frame_check']}\n")
            rc = 1
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    if rc:
        sys.exit(rc)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=int(os.environ.get("WORLD_SIZE", "1")))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="train_1m_1080p")
    ap.add_argument("--splats", type=int, default=0, help="override the workload's splat count (debug)")
    ap.add_argument("--value-depth", type=int, default=3, choices=[3, 4], help="tickets kept open in the device-resident timing loop")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the oracle legs (parity block + cpu_baseline)")
    ap.add_argument("--no-other-configs", action="store_true", help="N = 1: time only the headline configuration")
    ap.add_argument("--parallel", default="auto", choices=["auto", "frames", "tiles"],
                    help="N > 1: `frames` = every rank renders every N-th frame from its own replica (weak scaling, default); "
                         "`tiles` = one frame sharded by screen bin columns + tile exchange (strong scaling, default for the 80 M scene)")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                    help="multi-GPU frame exchange: fused raster + NVLink peer stores (default) or NCCL all-gather of tiles")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the RGBA8 frame of the last timed step of the headline configuration (as float32) to "
                         "DIR/<name>.npy, at most 64 MB: a seeded sample of the pixels when the frame is larger")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm shades only a band of rows per step; use it with --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
