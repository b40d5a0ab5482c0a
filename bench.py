#!/usr/bin/env python3
"""bench.py — Mray/s of the B200 path-tracing hot path on BASELINE.json's configs[1]
(hexagon_room.json, 1920x1080, 256 spp, quaternary_sah BVH), at 1/2/4/8 GPUs.

A "step" is one complete render of the frame: ray generation, wavefront loop (extend / shade /
shadow / regenerate) until every path has terminated, film resolve. Rays = closest-hit queries
(extension + shadow), counted by the kernels themselves.

  value      whole-job Mray/s with the scene resident in HBM and the framebuffer left in HBM; device
             time from CUDA events on the launching stream (library events around the render, torch
             events around the NCCL all-gather), max over ranks.
  e2e        same metric through the host-buffer C-ABI call: scene upload (H2D) + render + framebuffer
             D2H into pinned host memory inside the timed region (wall clock between synchronisations).
  roofline   the traversal kernel (k_extend): algorithmic bytes (SURVEY.md §8d: 48 B/ray + 32 B per
             box test + 48 B per primitive test, counted by the kernel) / its CUDA-event time, PLUS what
             this run measured in a non-timed ncu epilogue over the same kernels: DRAM bytes (traffic,
             dram_gbs) and FP64 thread-instructions against the FP64 issue rate measured in the run.
  secondary  the same measurements on BASELINE config 3's scene (spaceship, 457 k triangles) at 64 spp.
  cpu_baseline / --impl reference
             the UNMODIFIED reference (oracle/_ref, best of {hw, hw/2, ...} host threads) on a bounded
             sample of the same workload: the SAME full frame at a REDUCED sample count (1 spp on the
             driver's box for C2; rays/s does not depend on spp) - printed in `sample`.

Multi-GPU: rows are sharded interleaved (rank r renders rows r, r+N, ...; the same pixels as the
single-GPU image), the scene is replicated; the film resolve of every rank stores its rows straight
into the float3 frame of every rank (peer memory over NVLink, mcrt_render_rows_strided_peers), one
barrier per step. Total work is fixed as N grows ("strong").
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # id: (pack, reference scene json, reference overrides)
    "c2": ("bench_data/c2_hexagon_room.mcrtpack", "hexagon_room.json",
           dict(width=1920, height=1080, sqrtspp=16, bvh_type="quaternary_sah"),
           "hexagon_room.json 1920x1080 256spp quaternary_sah"),
    "c1": ("bench_data/c1_hexagon_room_diffuse.mcrtpack", "hexagon_room_diffuse.json",
           dict(width=256, height=256, sqrtspp=2, bvh_type="binary_sah", bins_per_axis=16),
           "hexagon_room_diffuse.json 256x256 4spp binary_sah"),
    # OBJ scenes: packs written by `python tools/validate_big.py make` (git-ignored, 35-81 MB); the camera is
    # resized to the BASELINE configuration
    "c3": ("bench_data/v3_spaceship.mcrtpack.xz", "spaceship.json",
           dict(width=1920, height=1080, sqrtspp=32),
           "spaceship.json 1920x1080 1024spp quaternary_sah"),
    # photon-mapped (PhotonMapper::sampleRay): the photon pass (1e6 emissions x caustic_factor 10, all on the GPU) runs
    # once before the timed steps; sqrtspp 23 = 529 spp, the nearest square to the 512 spp of BASELINE config 4
    "c4": ("bench_data/v4_water_caustics.mcrtpack.xz", "water_caustics.json",
           dict(width=1024, height=1024, sqrtspp=23, photon_map=dict(emissions=1e6, caustic_factor=10.0, k_nearest_photons=50)),
           "water_caustics.json 1024x1024 529spp photon_map 1e6 emissions k=50"),
    "c5": ("bench_data/v5_lego_bulldozer.mcrtpack.xz", "lego_bulldozer.json",
           dict(width=3840, height=2160, sqrtspp=64),
           "lego_bulldozer.json 3840x2160 4096spp quaternary_sah"),
}

METRIC = "Mray/s (primary+shadow+bounce)"


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()  # exact PID we started
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def traversal_bytes(rays, box, prim):
    return 48.0 * rays + 32.0 * box + 48.0 * prim


DUMP_LIMIT_BYTES = 64 << 20


def write_outputs(out_dir, frame):
    """--dump-outputs: the frame of the last timed step as out_dir/image.npy ([H, W, 3], float32 or float64 as rendered), so
    that two builds can be compared output for output. A frame over 64 MB is replaced by a fixed, seeded sample of its pixels:
    image_sample.npy [n, 3] and their flat pixel indices, image_sample_index.npy (float64)."""
    os.makedirs(out_dir, exist_ok=True)
    frame = np.ascontiguousarray(frame)
    assert frame.dtype in (np.float32, np.float64), frame.dtype
    if frame.nbytes <= DUMP_LIMIT_BYTES:
        np.save(os.path.join(out_dir, "image.npy"), frame)
        return
    pixels = frame.reshape(-1, 3)
    n = DUMP_LIMIT_BYTES // (3 * pixels.itemsize + 8)
    idx = np.sort(np.random.default_rng(0).choice(len(pixels), n, replace=False))
    np.save(os.path.join(out_dir, "image_sample.npy"), pixels[idx])
    np.save(os.path.join(out_dir, "image_sample_index.npy"), idx.astype(np.float64))


# ------------------------------------------------------------------------------------- reference arm
def reference_sample(workload, seconds_target, threads=-1):
    """The unmodified reference on a bounded sample of the workload: the SAME frame (scene, camera,
    resolution, BVH) at a reduced sample count, sized from a 1-spp calibration render so that one
    sample render takes about `seconds_target`. Rays/s does not depend on spp (every sample is an
    independent path), and the full frame keeps all 2040 32x32 buckets so every host thread has
    work. Returns (scene handle, threads used, sqrtspp)."""
    from oracle import ref
    _, scene_json, overrides, _ = WORKLOADS[workload]
    ref.set_seed(0x12345678)
    photon = overrides.get("photon_map")
    overrides = {k: v for k, v in overrides.items() if k != "photon_map"}
    if photon:
        overrides = dict(overrides, emissions=photon["emissions"])
    cal = ref.RefScene(scene_json, dict(overrides, sqrtspp=1), photon_map=bool(photon))
    hw = ref.lib().ref_hardware_threads()
    # The reference takes its thread count from std::thread::hardware_concurrency (integrator.cpp:20-23).
    # On hosts where that exceeds the cores this container may use it oversubscribes badly, so the
    # baseline is given the best of {hw, hw/2, hw/4, ...} threads (1-spp calibration renders).
    candidates = [threads] if threads >= 1 else sorted({max(1, hw >> k) for k in range(0, 5)}, reverse=True)
    best = None
    for t in candidates:
        _, sec, rays, _ = cal.render(threads=t)
        if best is None or rays / sec > best[1]:
            best = (t, rays / max(sec, 1e-6), rays)
    cal.close()
    cores, rate, rays = best
    k = int(max(1, min(overrides["sqrtspp"], round((seconds_target * rate / max(rays, 1)) ** 0.5))))
    s = ref.RefScene(scene_json, dict(overrides, sqrtspp=k), photon_map=bool(photon))
    s.best_threads = cores
    return s, cores, k


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    _, _, _, label = WORKLOADS[args.workload]
    per_step = args.baseline_seconds if args.baseline_seconds > 0 else max(2.0, min(20.0, 120.0 / max(1, args.steps + args.warmup)))
    s, cores, k = reference_sample(args.workload, per_step)
    for _ in range(args.warmup):
        s.render(threads=cores)
    tot_rays, tot_sec = 0, 0.0
    for _ in range(args.steps):
        img, sec, rays, _ = s.render(threads=cores)
        tot_rays += rays; tot_sec += sec
    if args.dump_outputs:
        write_outputs(args.dump_outputs, img)
    value = tot_rays / tot_sec / 1e6
    sample = (f"full {s.width}x{s.height} frame at {k * k} spp instead of {WORKLOADS[args.workload][2]['sqrtspp'] ** 2} "
              f"({tot_rays // max(1, args.steps)} rays/step), unmodified reference, best of {{hw, hw/2, ...}} = {cores} threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "Mray/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_sec / max(1, args.steps),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "reference scene (vendored hexagon_room.json), fixed sampler seed",
        "config": {"workload": label, "sample": sample},
        "cpu_baseline": {"value": value, "unit": "Mray/s", "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": "Mray/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------ GPU arm
NCU_METRICS = ["gpu__time_duration.sum", "dram__bytes_read.sum", "dram__bytes_write.sum",
               "smsp__sass_thread_inst_executed_op_dadd_pred_on.sum", "smsp__sass_thread_inst_executed_op_dmul_pred_on.sum",
               "smsp__sass_thread_inst_executed_op_dfma_pred_on.sum", "smsp__thread_inst_executed.sum", "smsp__inst_executed.sum"]


def child_render(args):
    """One untimed render of the workload at a reduced sample count; prints its counters as JSON. Run under ncu
    by profile_kernels() - nothing measured here is a bench value."""
    m = importlib.import_module("monte-carlo-ray-tracer_b200")
    pack, _, ov, _ = WORKLOADS[args.workload]
    scene = m.Scene.from_pack(os.path.join(ROOT, pack))
    cam = scene.cameras()[0].resized(ov["width"], ov["height"], args.sqrtspp or 2)
    prec = m.PRECISION_F64 if args.precision == "f64" else m.PRECISION_F32
    if ov.get("photon_map"):
        pe = scene.extra["photon_emit_params"]; ph = ov["photon_map"]
        pt = m.PhotonMapper(scene, device=0, precision=prec, global_seed=0x12345678,
                            emit=dict(emissions=int(ph["emissions"]), caustic_factor=ph["caustic_factor"], max_photons_per_octree_leaf=int(pe[2]),
                                      k_nearest_photons=ph["k_nearest_photons"], scene_bounds=pe[3:9]))
    else:
        pt = m.PathTracer(scene, device=0, precision=prec, global_seed=0x12345678)
    pt.set_option("pool_paths", args.pool if args.pool else float(1 << 25))
    import torch
    out = torch.zeros((cam.height, cam.width, 3), dtype=torch.float64, device="cuda:0")
    st = pt.render_rows_dev(cam, out.data_ptr())
    print("CHILD_STATS " + json.dumps(st), flush=True)
    pt.close()
    return 0


def profile_kernels(args, workload, sqrtspp):
    """Non-timed epilogue: the same code path under `ncu` at a reduced sample count, every launch of the stage
    kernels counted once: DRAM bytes, FP64 thread-instructions, active lanes per instruction, per kernel.
    -> {kernel: {...}} with per-ray figures, or {"unavailable": why}."""
    import shutil
    if not shutil.which("ncu"):
        return {"unavailable": "ncu not on PATH"}
    cmd = ["ncu", "--metrics", ",".join(NCU_METRICS), "--clock-control", "none", "-k", "regex:k_extend|k_shade|k_shadow|k_knn",
           "--print-units", "base", "--csv", sys.executable, os.path.abspath(__file__), "--child-render", "--workload", workload, "--sqrtspp", str(sqrtspp),
           "--precision", args.precision] + (["--pool", str(args.pool)] if args.pool else [])
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "0")))
    except Exception as e:
        return {"unavailable": f"{type(e).__name__}: {str(e)[:160]}"}
    out = parse_ncu_output(r.stdout)
    if "unavailable" in out:
        out["unavailable"] += " | " + (r.stderr or "")[-160:].replace("\n", " ")
        return out
    out["sample"] = f"{workload} at {sqrtspp * sqrtspp} spp under ncu (all launches of the stage kernels, each counted once)"
    return out


def parse_ncu_output(text):
    """`ncu --csv` rows + the child's CHILD_STATS line -> per-kernel, per-unit figures (see profile_kernels)."""
    import csv
    import io
    stats = None
    rows = []
    for ln in text.splitlines():
        if ln.startswith("CHILD_STATS "):
            stats = json.loads(ln[len("CHILD_STATS "):])
        elif ln.startswith('"'):
            rows.append(ln)
    if stats is None or len(rows) < 2:
        return {"unavailable": "ncu produced no counters: " + text[-200:].replace("\n", " ")}
    rd = list(csv.reader(io.StringIO("\n".join(rows))))
    hdr = rd[0]
    ik, im, iv = hdr.index("Kernel Name"), hdr.index("Metric Name"), hdr.index("Metric Value")
    iu = hdr.index("Metric Unit") if "Metric Unit" in hdr else None
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    agg = {}
    for row in rd[1:]:
        if len(row) <= iv:
            continue
        name = row[ik]
        key = "k_shade_key" if "k_shade_key" in name else next((k for k in ("k_extend", "k_shadow", "k_shade", "k_knn") if k in name), None)
        if key is None:
            continue
        try:
            v = float(row[iv].replace(",", ""))
        except ValueError:
            continue
        if iu is not None and row[im].startswith("dram__bytes"):
            v *= scale.get(row[iu], 1.0)           # ncu prints byte counts in auto-scaled units unless told otherwise
        a = agg.setdefault(key, {"launches": 0})
        a[row[im]] = a.get(row[im], 0.0) + v
        if row[im] == "gpu__time_duration.sum":
            a["launches"] += 1
    units = {"k_extend": stats["extension_rays"], "k_shadow": stats["shadow_rays"], "k_shade": stats["extension_rays"], "k_knn": max(1, stats["knn_queries"])}
    out = {}
    for k, a in agg.items():
        if k not in units or not units[k]:
            continue
        n = float(units[k])
        fp64 = sum(a.get(f"smsp__sass_thread_inst_executed_op_{op}_pred_on.sum", 0.0) for op in ("dadd", "dmul", "dfma"))
        out[k] = {"launches": a["launches"], "dram_bytes_per_unit": (a.get("dram__bytes_read.sum", 0.0) + a.get("dram__bytes_write.sum", 0.0)) / n,
                  "fp64_thread_inst_per_unit": fp64 / n,
                  "lanes_per_inst": a.get("smsp__thread_inst_executed.sum", 0.0) / max(1.0, a.get("smsp__inst_executed.sum", 1.0)),
                  "unit": "query" if k == "k_knn" else "ray"}
    return out


def measure(env, args, workload, steps, warmup, sqrtspp_override=0, profile=True, dump_dir=None):
    """Times `steps` renders of `workload` on this job's GPUs; with `dump_dir`, rank 0 writes the frame of the last timed
    step there (write_outputs). -> result dict on rank 0 (None elsewhere)."""
    torch, dist, m, mdist = env["torch"], env["dist"], env["m"], env["mdist"]
    rank, local_rank, world = env["rank"], env["local_rank"], env["world"]
    pack, _, ov, label = WORKLOADS[workload]
    if not os.path.exists(os.path.join(ROOT, pack)):
        raise SystemExit(f"bench.py: {pack} is missing - generate it with `python tools/validate_big.py make` where /root/reference exists")
    scene = m.Scene.from_pack(os.path.join(ROOT, pack))
    cam = scene.cameras()[0].resized(ov["width"], ov["height"], sqrtspp_override or ov["sqrtspp"])
    precision = m.PRECISION_F64 if args.precision == "f64" else m.PRECISION_F32
    photon = ov.get("photon_map")
    photon_pass = None
    if photon:
        pe = scene.extra["photon_emit_params"]
        pt = m.PhotonMapper(scene, device=local_rank, precision=precision, global_seed=0x12345678)   # maps of the pack: replaced below
        kw = dict(emissions=int(photon["emissions"]), caustic_factor=photon["caustic_factor"], max_photons_per_octree_leaf=int(pe[2]),
                  k_nearest_photons=photon["k_nearest_photons"], scene_bounds=pe[3:9])
        t0 = time.perf_counter()
        n_c, n_g = pt.emit_sharded(rank, world, **kw) if world > 1 else pt.emit(**kw)
        torch.cuda.synchronize()
        photon_pass = {"emission_gpu_ms": pt.last_stats["gpu_ms_total"], "octree_build_gpu_ms": pt.last_stats["gpu_ms_knn"],
                       "photon_rays": pt.last_stats["extension_rays"], "caustic_photons": int(n_c), "global_photons": int(n_g),
                       "wall_s": time.perf_counter() - t0, "sharded_over": world}
    else:
        pt = m.PathTracer(scene, device=local_rank, precision=precision, global_seed=0x12345678)
    pt.set_option("pool_paths", args.pool if args.pool else float(1 << 25))   # 32 Mi paths in flight (19 GB of HBM: 576 B per path in float64)
    pt.set_option("stage_timing", 1)
    W, H = cam.width, cam.height
    dev = torch.device("cuda", local_rank)
    # every rank holds the whole float3 frame; each rank's resolve kernel stores its rows into all of them (NVLink)
    frames = mdist.PeerFrames(pt, rank, world, H, W, float32=True, device=dev)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def step():
        st = frames.render(cam)       # returns after this rank's kernels (incl. the peer stores) have completed
        frames.barrier()              # every rank's rows are in every frame
        return st["gpu_ms_total"], st

    for _ in range(warmup):
        step()
    sampler = ClockSampler(local_rank)
    sync_all()
    sampler.start()
    wall0 = time.perf_counter()
    dev_ms, stats = 0.0, []
    for _ in range(steps):
        ms, st = step()
        dev_ms += ms
        stats.append(st)
    sync_all()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop()
    # copied before the e2e leg, which renders into the same frames when N > 1
    last_frame = frames.tensor().cpu().numpy() if dump_dir and rank == 0 else None

    # ---- e2e: host buffers in, host buffers out. N=1: the plain C-ABI call mcrt_scene_upload + mcrt_render_rows
    # (float64 frame to the host). N>1: scene upload + sharded render + rank 0 reads the assembled float3 frame.
    e2e_steps = steps
    host64 = torch.empty((H, W, 3), dtype=torch.float64).pin_memory() if world == 1 else None
    host32 = torch.empty((H, W, 3), dtype=torch.float32).pin_memory() if world > 1 else None
    frame_t = frames.tensor() if world > 1 else None

    def e2e_step():
        h2d = pt.upload_scene() + 144  # scene arrays + camera record
        if world == 1:
            pt.render_rows(cam, 0, H, out=host64.numpy())
            return h2d, pt.last_stats
        st = frames.render(cam)
        frames.barrier()
        if rank == 0:
            host32.copy_(frame_t, non_blocking=False)
        return h2d, st

    h2d_bytes, e2e_rays, e2e_wall = 0, 0, 0.0
    if not args.no_e2e:
        e2e_step()
        sync_all()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            h2d_bytes, st = e2e_step()
            e2e_rays += st["extension_rays"] + st["shadow_rays"]
        sync_all()
        e2e_wall = time.perf_counter() - t0
    d2h_bytes = H * W * 3 * (8 if world == 1 else 4)

    def allreduce(x, op):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return float(t.item())

    SUM, MAX = (dist.ReduceOp.SUM, dist.ReduceOp.MAX) if world > 1 else (None, None)
    rays_local = sum(s["extension_rays"] + s["shadow_rays"] for s in stats)
    rays_total = allreduce(float(rays_local), SUM)
    dev_ms_max = allreduce(dev_ms, MAX)
    dev_ms_mean = allreduce(dev_ms, SUM) / world
    wall_max = allreduce(wall, MAX)
    e2e_rays_total = allreduce(float(e2e_rays), SUM)
    e2e_wall_max = allreduce(e2e_wall, MAX)
    launches = allreduce(float(sum(s["kernel_launches"] for s in stats)), SUM)
    fp64_peak = pt.fp64_peak() if args.precision == "f64" else None

    # ---- the traversal kernel (rank 0's launches)
    ext_rays = sum(s["extension_rays"] for s in stats)
    sh_rays = sum(s["shadow_rays"] for s in stats)
    ext_box = sum(s["box_tests"] - s["shadow_box_tests"] for s in stats)
    ext_prim = sum(s["prim_tests"] - s["shadow_prim_tests"] for s in stats)
    ext_ms = sum(s["gpu_ms_extend"] for s in stats)
    ext_launches = sum(s["extend_launches"] for s in stats)
    sh_ms = sum(s["gpu_ms_shadow"] for s in stats)
    shade_ms = sum(s["gpu_ms_shade"] for s in stats)
    gen_ms = sum(s["gpu_ms_generate"] for s in stats)
    replayed = sum(s["replayed_rays"] for s in stats)
    knn_queries = sum(s["knn_queries"] for s in stats)
    knn_ms = sum(s["gpu_ms_knn"] for s in stats)
    pt.close()
    frames_bytes = frames.nbytes
    # (the frames stay mapped until the process ends: closing them needs another barrier and buys nothing here)

    if rank != 0:
        return None
    if last_frame is not None:
        write_outputs(dump_dir, last_frame)
    peak, peak_src = measured_peaks()
    alg_bytes = traversal_bytes(ext_rays, ext_box, ext_prim)
    achieved = alg_bytes / (ext_ms * 1e-3) / 1e9 if ext_ms > 0 else 0.0
    scene_bytes = int(pt.h2d_bytes)
    prof = profile_kernels(args, workload, 3 if W * H >= 1000000 else 8) if (profile and world == 1) else {"unavailable": "profiled at N=1 only"}
    pe = prof.get("k_extend") if isinstance(prof, dict) else None
    avg_launch_ms = ext_ms / max(1, ext_launches)
    rays_per_launch = ext_rays / max(1, ext_launches)
    roofline = {
        "kernel": "k_extend<%s>%s" % ("double" if args.precision == "f64" else "float", " (order-free search, replay of ambiguous rays)" if args.precision == "f64" else ""),
        "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
        "algorithmic_bytes": "SURVEY.md 8(d): 48 B/ray + 32 B per box test + 48 B per primitive test, counted by the kernel",
        "algorithmic_bytes_per_launch": alg_bytes / max(1, ext_launches), "bytes_per_ray": alg_bytes / max(1, ext_rays),
        "avg_launch_ms": avg_launch_ms, "launches": ext_launches,
        # measured in this run (ncu epilogue over the same kernels at a reduced sample count), scaled by rays:
        "traffic": pe["dram_bytes_per_unit"] * rays_per_launch if pe else None,
        "dram_gbs": pe["dram_bytes_per_unit"] * ext_rays / (ext_ms * 1e-3) / 1e9 if pe and ext_ms > 0 else None,
        "scene_bytes": scene_bytes,
        "note": ("the scene (%d bytes) is served from L1/L2, so `frac` counts cache hits as HBM bytes: it measures box/primitive-test throughput, "
                 "may exceed 1 and is not the binding roofline; dram_gbs is what crosses HBM, fp64 is the issue-rate bound" % scene_bytes)
                if scene_bytes < 126e6 else "scene larger than L2",
    }
    if pe and ext_ms > 0:
        roofline["dram_frac"] = roofline["dram_gbs"] / peak
        roofline["lanes_per_inst"] = pe["lanes_per_inst"]
        if fp64_peak:
            rate = pe["fp64_thread_inst_per_unit"] * ext_rays / (ext_ms * 1e-3)
            roofline["fp64"] = {"achieved": rate / 1e12, "peak": fp64_peak / 1e12, "unit": "T thread-inst/s (DADD+DMUL+DFMA)", "frac": rate / fp64_peak,
                                "inst_per_ray": pe["fp64_thread_inst_per_unit"], "peak_source": "measured in this run (mcrt_fp64_peak: independent DFMA chains)"}
    if isinstance(prof, dict) and "unavailable" in prof:
        roofline["profile_unavailable"] = prof["unavailable"]
    value = rays_total / (dev_ms_max * 1e-3) / 1e6
    result = {
        "metric": METRIC, "value": value, "unit": "Mray/s", "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": dev_ms_max / steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": args.precision,
        "data": "reference scene flattened by the reference's own loader / BVH builder (scene pack), fixed sampler seed",
        "config": {"workload": label if not sqrtspp_override else f"{label} [at {sqrtspp_override ** 2} spp]",
                   "paths_per_step": W * H * cam.sqrtspp ** 2, "rays_per_step": rays_total / steps,
                   "parallelism": (f"rows interleaved over {world} GPUs, scene replicated; each rank's film resolve stores its rows into every rank's "
                                   f"float3 frame over NVLink (CUDA IPC peer memory), one barrier per step") if world > 1 else "1 GPU",
                   "l2": "per-step working set (32 Mi-path pool, 19 GB of queues) exceeds the 126 MB L2; see roofline.note for the scene arrays",
                   "mode": "parity (float64 primitive tests and shading in the reference's operation order, --fmad=false)" if args.precision == "f64" else "fast (float32)"},
        "wall_ms_per_step": 1e3 * wall_max / steps,
        "rank_imbalance": {"max_over_mean_gpu_ms": dev_ms_max / max(1e-9, dev_ms_mean)},
        "e2e": {"value": (e2e_rays_total / e2e_wall_max / 1e6) if e2e_wall_max > 0 else None, "unit": "Mray/s",
                "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(d2h_bytes),
                "steps": e2e_steps, "timing": "wall clock between synchronisations, max over ranks"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "stage_ms_per_step": {"extend": ext_ms / steps, "shade(+class sort)": shade_ms / steps, "shadow": sh_ms / steps, "generate+advance+sort": gen_ms / steps},
        "rays": {"extension_per_step": ext_rays / steps, "shadow_per_step": sh_rays / steps, "replayed_in_reference_order": replayed / steps,
                 "box_tests_per_ray": (ext_box) / max(1, ext_rays), "prim_tests_per_ray": ext_prim / max(1, ext_rays)},
        "kernels": {k: v for k, v in prof.items() if k != "k_extend"} if isinstance(prof, dict) else None,
    }
    if photon:
        result["photon_pass"] = photon_pass
        result["knn"] = {"queries_per_step": knn_queries / steps, "mquery_per_s_in_kernel": knn_queries / max(1e-9, knn_ms) / 1e3,
                         "mquery_per_s_whole_step": knn_queries / (dev_ms * 1e-3) / 1e6, "k_knn_ms_per_step": knn_ms / steps,
                         "algorithmic_bytes_per_query": 12400, "hbm_frac_algorithmic": 12400.0 * knn_queries / max(1e-9, knn_ms * 1e-3) / 1e9 / peak}
    return result


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU path)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    env = {"torch": torch, "dist": dist, "rank": rank, "local_rank": local_rank, "world": world,
           "m": importlib.import_module("monte-carlo-ray-tracer_b200"),
           "mdist": importlib.import_module("monte-carlo-ray-tracer_b200.distributed")}

    line = measure(env, args, args.workload, args.steps, args.warmup, args.sqrtspp, profile=not args.no_profile, dump_dir=args.dump_outputs)
    # secondary block: the 457 k-triangle spaceship (BASELINE config 3) at a sample count that keeps the default run short
    secondary = None
    sec_pack = os.path.join(ROOT, WORKLOADS["c3"][0])
    if args.workload == "c2" and not args.no_secondary and not args.sqrtspp and os.path.exists(sec_pack):
        secondary = measure(env, args, "c3", args.steps, args.warmup, 8, profile=not args.no_profile)

    if rank == 0:
        if secondary is not None:
            line["secondary"] = {k: secondary[k] for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "config", "e2e", "roofline",
                                                          "stage_ms_per_step", "rays", "kernels", "rank_imbalance", "gpu_launches")}
        if world == 1 and not args.no_cpu_baseline:
            # The reference arm runs in a child process: the reference aborts on a scene whose assets are
            # missing (e.g. OBJ scenes on a box without /root/reference), and that must not take the
            # measured arm down with it.
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", args.workload,
                                    "--steps", "1", "--warmup", "0", "--sqrtspp", "1", "--baseline-seconds", "15"],
                                   capture_output=True, text=True, timeout=900)
                ref_line = json.loads(r.stdout.strip().splitlines()[-1])
                line["cpu_baseline"] = ref_line["cpu_baseline"]
            except Exception as e:  # the oracle is test infrastructure; report, don't hide
                line["cpu_baseline"] = {"value": None, "unit": "Mray/s", "cores": 0, "kind": "reference",
                                        "sample": f"unavailable on this box: {type(e).__name__}: {str(e)[:200]}"}
        print(json.dumps(line), flush=True)

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="f64", choices=["f64", "f32"])
    ap.add_argument("--sqrtspp", type=int, default=0, help="override samples (debug only; invalidates the config)")
    ap.add_argument("--pool", type=float, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true", help="skip the ncu epilogue (measured DRAM traffic / FP64 counts)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the spaceship block")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer end-to-end leg (long single-purpose runs only)")
    ap.add_argument("--child-render", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--baseline-seconds", type=float, default=0.0, help="reference arm: target seconds per step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frame of the last timed step to DIR/image.npy (inputs are fixed: same arguments, same frame)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and not args.sqrtspp and args.workload == "c2":   # the contract's W >= 3 for the headline workload
        args.warmup = 3
    if args.child_render:
        return child_render(args)
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_gpu_arm(args)


if __name__ == "__main__":
    sys.exit(main())
