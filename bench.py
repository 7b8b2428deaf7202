#!/usr/bin/env python
"""bench.py — frames/s of the per-volume fusion+raycast loop on synthetic KITTI-shaped streams.

    python bench.py --gpus N --steps K --warmup W            (own arm, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K ...  (reference arm: CPU, rank 0 only)

A step is one frame through {AllocateSceneFromDepth, IntegrateIntoScene, CreateExpectedDepths,
CreateICPMaps (raycast), Decay(partial)} on one ITMScene volume (BASELINE.json configs[1]; SURVEY 8d).
value  = frames/s with the frames already resident in HBM (whole job: all ranks' frames / max time)
e2e    = frames/s through b200_host_frame_submit/_wait (host buffers in, host image out): every frame's
         depth+RGB are copied from pinned host memory and its grey raycast image is copied back inside the
         timed region; the copies of neighbouring frames overlap the kernels (two staging slots)
roofline = IntegrateIntoScene: algorithmic bytes (8224 B per integrated block + w*h*8 B of images
         per launch) / mean launch duration from CUDA events around every launch of the timed region
cpu_baseline = the CPU oracle (oracle/tsdf_oracle.c, OpenMP at the reference's own pragma sites)
         timed on this box's host cores on a bounded sample of the same stream.
N > 1: one independent volume per rank (weak scaling; no data-path collective inside fusion); the
per-volume raycast image is gathered to rank 0 over NCCL every frame (SURVEY 8e).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from dynslam_b200 import synth  # noqa: E402

METRIC = "frames/sec TSDF fusion+raycast at KITTI 1242x375; Mvoxels/s integrated"
NUM_BLOCKS, NUM_BUCKETS, EXCESS = 0x60000, 0x100000, 0x80000   # ITMLibSettings.cpp:115, ITMLibDefines.h:42-53
DECAY = (1, 200)                                                # --max_decay_weight=1 --min_decay_age=200 (DynSLAMGUI.cpp:38-40)
BYTES_PER_BLOCK = 8192 + 32                                     # SURVEY 8d


def log(*a):
    print(*a, file=sys.stderr, flush=True)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.proc = index, [], False, None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def pause(self, on):
        """SIGSTOP / SIGCONT nvidia-smi: its 20 ms polling was measured to stall the driver for 50-70 ms now and then, which a
        host-synchronous loop (the e2e phases) sees in full; the clocks are only needed for the device-timed region."""
        import signal
        if self.proc and self.proc.poll() is None:
            try:
                self.proc.send_signal(signal.SIGSTOP if on else signal.SIGCONT)
            except Exception:
                pass

    def stop(self):
        self.stop_flag = True
        if self.proc:
            self.pause(False)
            self.proc.terminate()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def frame_gaps(marks):
    """Host-side spacing of consecutive pipelined submissions (ms): median / max / index of the max — exposes one-off stalls."""
    if len(marks) < 3:
        return None
    d = np.diff(np.asarray(marks)) * 1000.0
    return {"median": float(np.median(d)), "max": float(d.max()), "argmax": int(d.argmax()), "n": int(d.size)}


def gen_frames(seed, first, count, length_m):
    scene = synth.StreetScene(seed=seed, length_m=length_m)
    out = []
    for f in range(first, first + count):
        depth, rgb, M, proj = synth.kitti_frame(scene, f)
        out.append((depth, rgb, M, proj))
    return out


def gen_frames_parallel(seed, first, count, length_m, workers):
    if count <= 0:
        return []
    if workers <= 1 or count < 8:
        return gen_frames(seed, first, count, length_m)
    import multiprocessing as mp
    chunk = (count + workers - 1) // workers
    jobs = [(seed, first + i * chunk, min(chunk, count - i * chunk), length_m) for i in range(workers) if i * chunk < count]
    with mp.get_context("fork").Pool(len(jobs)) as pool:
        parts = pool.starmap(gen_frames, jobs)
    return [f for p in parts for f in p]


def gen_frames_cars(seed, first, count, length_m, ncars):
    """configs[2] frames: the street of `seed` with `ncars` followed cars; (depth, rgb, M, proj, [mask or None per car])"""
    scene = synth.StreetScene(seed=seed, length_m=length_m)
    cars = [synth.FollowedCar(i, seed=3) for i in range(ncars)]
    proj = synth.kitti_intrinsics()
    out = []
    for f in range(first, first + count):
        M = synth.kitti_pose(f)
        depth, rgb, ident = scene.render(M, synth.KITTI_W, synth.KITTI_H, float(proj[0]), float(proj[1]), float(proj[2]), float(proj[3]),
                                         extra_boxes=[c.box(f) for c in cars], want_ids=True)
        out.append((depth, rgb, M, proj, [synth.silhouette_mask(ident, i) for i in range(ncars)]))
    return out


def gen_frames_cars_parallel(seed, first, count, length_m, ncars, workers):
    if workers <= 1 or count < 8:
        return gen_frames_cars(seed, first, count, length_m, ncars)
    import multiprocessing as mp
    chunk = (count + workers - 1) // workers
    jobs = [(seed, first + i * chunk, min(chunk, count - i * chunk), length_m, ncars) for i in range(workers) if i * chunk < count]
    with mp.get_context("fork").Pool(len(jobs)) as pool:
        parts = pool.starmap(gen_frames_cars, jobs)
    return [f for p in parts for f in p]


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    p = os.path.join(ROOT, "profiles", "integrate_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("dram_bytes_per_launch")
        except Exception:
            return None
    return None


# --------------------------------------------------------------------------------------------------
# CPU oracle leg (cpu_baseline of the own arm and the whole --impl reference arm)
# --------------------------------------------------------------------------------------------------
def base_config(preroll):
    """the workload keys both arms report identically (the driver compares the two lines' config)"""
    return {"workload": "KITTI-odometry-06-shaped 1242x375 static-map fusion+raycast loop (configs[1]); one volume per GPU",
            "voxel_m": 0.05, "mu_m": 0.75, "maxW": 50, "blocks": NUM_BLOCKS, "buckets": NUM_BUCKETS, "excess": EXCESS,
            "decay": {"maxWeight": DECAY[0], "minAge": DECAY[1]}, "preroll_frames": preroll}


def cpu_run(seed, preroll, warmup, steps, passes=1, threads=None):
    """The CPU oracle on this box's host cores (OpenMP at the reference's own pragma sites: per-pixel marking, per-block
    integration, per-pixel raycast; the table sweeps stay serial as in the reference). Same stream, same pre-roll as the GPU
    arm (the decay queue is live), a FIXED thread count (no calibration: VERDICT r1 weak #2), `passes` consecutive passes of
    `steps` frames; the reported figure is the median pass."""
    from tests import hostlib as H
    L = H.oracle()
    ncpu = os.cpu_count() or 1
    # fixed, stated: 32 threads (or every core of a smaller box). More does not help the oracle: its table sweeps are serial, as in
    # the reference, and the per-pixel regions are short — measured on the 128-thread B200 host: 30 frames/s at 32 threads, 5 at 128.
    threads = threads or min(32, ncpu)
    L.oracle_set_threads(threads)
    vol = H.HostVolume(NUM_BLOCKS, NUM_BUCKETS, EXCESS, synth.KITTI_W, synth.KITTI_H)
    n = preroll + warmup + steps * passes
    frames = gen_frames_parallel(seed, 0, n, n * 0.8 + 60.0, min(16, ncpu))

    def one(fr):
        depth, rgb, M, proj = fr
        v = H.make_view(depth, rgb, M, proj)
        L.oracle_allocate_from_depth(vol.engine, C.byref(vol.scene), C.byref(vol.rs), C.byref(v), 0, 1)
        L.oracle_integrate(vol.engine, C.byref(vol.scene), C.byref(vol.rs), C.byref(v), 1)
        nb = L.oracle_integrated_blocks(vol.engine)
        cam = H.make_camera(M, proj)
        L.oracle_expected_depths(C.byref(vol.scene), C.byref(vol.rs), C.byref(cam))
        L.oracle_icp_maps(C.byref(vol.scene), C.byref(vol.rs), C.byref(v), H.vptr(vol.points), H.vptr(vol.normals), 1)
        L.oracle_decay(vol.engine, C.byref(vol.scene), C.byref(vol.rs), DECAY[0], DECAY[1], 0)
        return nb

    for fr in frames[:preroll + warmup]:
        one(fr)
    fps, vox_rate = [], []
    for p in range(passes):
        t0 = time.perf_counter()
        vox = 0
        for fr in frames[preroll + warmup + p * steps: preroll + warmup + (p + 1) * steps]:
            vox += one(fr) * 512
        dt = time.perf_counter() - t0
        fps.append(steps / dt)
        vox_rate.append(vox / dt / 1e6)
    med = float(np.median(fps))
    return {"fps": med, "passes_fps": fps, "spread": (max(fps) - min(fps)) / med if med > 0 else 0.0, "ms_per_step": 1000.0 / med if med > 0 else 0.0,
            "mvoxels_per_s": float(np.median(vox_rate)), "cores": L.oracle_num_threads(), "frames": steps, "passes": passes,
            "preroll": preroll, "visible_blocks": int(vol.rs.noVisibleBlocks), "decayed_blocks": int(L.oracle_decayed_block_count(vol.engine))}


def run_reference(args, rank, world):
    if rank != 0:
        return
    r = cpu_run(6, args.preroll, args.warmup, args.steps, passes=3)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["fps"], "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(base_config(args.preroll), l2="n/a (CPU arm)", integrate_impl="oracle/tsdf_oracle.c", parallelism=f"{r['cores']} OpenMP threads, 1 volume"),
        "mvoxels_per_s": r["mvoxels_per_s"], "passes_fps": r["passes_fps"], "spread": r["spread"],
        "visible_blocks": r["visible_blocks"], "decayed_blocks": r["decayed_blocks"],
        "cpu_baseline": {"value": r["fps"], "unit": "frames/s", "cores": r["cores"], "kind": "port",
                         "sample": f"median of {r['passes']} consecutive passes of {r['frames']} frames after a {r['preroll']}-frame pre-roll + "
                                   f"{args.warmup} warm-up frames of the same stream (decay queue live, as in the GPU arm), fixed at {r['cores']} "
                                   "threads; oracle/tsdf_oracle.c with OpenMP at the reference's pragma sites (the reference's own _CPU hash "
                                   "engines are commented out, SURVEY finding 1)"},
        "e2e": {"value": r["fps"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# parity of the TIMED state (VERDICT r1 #1): the frames bench.py pushed through the fused GPU path — pre-roll, warm-up and
# the timed steps — are replayed through the CPU oracle afterwards (outside every timed region) and the final hash table,
# free lists, visibility bytes, visible list, voxel array, ray points, ICP points and image are compared bit for bit.
# The oracle is used as the checker only (serial marking; OpenMP only over independent blocks / pixels).
# --------------------------------------------------------------------------------------------------
def gpu_snapshot(scene, rs, points):
    import torch
    torch.cuda.synchronize()
    g, r = scene.to_host(), rs.to_host()
    g.update(visType=r["visType"], visiblePos=r["visiblePos"], noVisibleBlocks=r["noVisibleBlocks"],
             raycastResult=rs.raycastResult.cpu().numpy(), raycastImage=rs.raycastImage.cpu().numpy(), points=points.cpu().numpy())
    return g


def parity_check(frames, n_frames, snap):
    from tests import hostlib as H
    L = H.oracle()
    t0 = time.perf_counter()
    vol = H.HostVolume(NUM_BLOCKS, NUM_BUCKETS, EXCESS, synth.KITTI_W, synth.KITTI_H)
    for depth, rgb, M, proj in frames[:n_frames]:
        v, cam = H.make_view(depth, rgb, M, proj), H.make_camera(M, proj)
        if L.oracle_allocate_from_depth(vol.engine, C.byref(vol.scene), C.byref(vol.rs), C.byref(v), 0, 0) != 0:
            return {"parity_checked": False, "why": "oracle ran out of blocks"}
        L.oracle_integrate(vol.engine, C.byref(vol.scene), C.byref(vol.rs), C.byref(v), 1)
        L.oracle_expected_depths(C.byref(vol.scene), C.byref(vol.rs), C.byref(cam))
        L.oracle_icp_maps(C.byref(vol.scene), C.byref(vol.rs), C.byref(v), H.vptr(vol.points), H.vptr(vol.normals), 1)
        L.oracle_decay(vol.engine, C.byref(vol.scene), C.byref(vol.rs), DECAY[0], DECAY[1], 0)
    nv = vol.rs.noVisibleBlocks
    pairs = [("hash", snap["hash"].tobytes(), vol.hash.tobytes()), ("voxels", snap["voxels"], vol.voxels),
             ("allocationList", snap["allocationList"], vol.allocationList), ("excessList", snap["excessList"], vol.excessList),
             ("entriesVisibleType", snap["visType"], vol.visType), ("visibleBlocks", snap["visiblePos"], vol.visiblePos[:max(nv, 0)]),
             ("raycastResult", snap["raycastResult"], vol.raycastResult.reshape(-1)),
             ("raycastImage", snap["raycastImage"], vol.raycastImage.reshape(-1)), ("points", snap["points"], vol.points.reshape(-1))]
    bad = []
    for name, a, b in pairs:
        if isinstance(a, bytes):
            # the 20-byte entries carry 2 padding bytes the reference leaves indeterminate: compare field by field
            ok = all(np.array_equal(snap["hash"][f], vol.hash[f]) for f in ("pos", "offset", "ptr", "allocatedTime"))
        else:
            a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
            ok = a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))
        if not ok:
            bad.append(name)
    counters_ok = (snap["lastFreeBlockId"] == vol.scene.lastFreeBlockId and snap["lastFreeExcessListId"] == vol.scene.lastFreeExcessListId
                   and snap["noVisibleBlocks"] == nv)
    if not counters_ok:
        bad.append("counters")
    return {"parity_checked": not bad, "frames_replayed": n_frames, "differing": bad,
            "compared": [p[0] for p in pairs] + ["counters"], "decayed_blocks_oracle": int(L.oracle_decayed_block_count(vol.engine)),
            "visible_blocks_oracle": int(nv), "allocated_blocks_oracle": int(NUM_BLOCKS - 1 - vol.scene.lastFreeBlockId),
            "oracle_seconds": time.perf_counter() - t0,
            "what": "bit-exact comparison of the GPU state right after the last timed step with the CPU oracle's after the same "
                    "frames (pre-roll + warm-up + timed), run after the timed region"}


# --------------------------------------------------------------------------------------------------
# the same stream through the REAL ITMLib objects (oracle/itm_harness.cpp): unmodified reference CUDA
# engines built for sm_100a vs. the B200 shim classes; pinned H2D of every frame inside the timing
# --------------------------------------------------------------------------------------------------
def run_itm_harness(preroll, timed, repeats=3):
    """scripts/harness_repeat.py in a FRESH process (no torch, nothing else has touched the CUDA allocator there): the reference's
    own engines `cudaMalloc` a copy of the visible list every frame and `cudaFree` it 200 frames later (Reco_CUDA.cu:302-317, :505),
    so their speed depends on the allocator's state — measured 126-1297 frames/s while the decay queue is still filling (every frame
    allocates, nothing is freed) against a stable 2 250 frames/s once it pops. The pre-roll therefore equals the own arm's (230 > minAge)."""
    so = os.path.join(ROOT, "oracle", "_ref", "libitmharness.so")
    if not os.path.exists(so):
        return {"error": "oracle/_ref/libitmharness.so not built"}
    cmd = [sys.executable, os.path.join(ROOT, "scripts", "harness_repeat.py"), str(preroll + timed), str(preroll), str(repeats)]
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    if p.returncode or not lines:
        return {"error": f"harness_repeat.py rc={p.returncode}: {p.stderr[-300:]}"}
    out = json.loads(lines[-1])
    out["what"] = ("per frame: pinned H2D of depth+RGB into the ITMView, then AllocateSceneFromDepth, IntegrateIntoScene, "
                   "CreateExpectedDepths, CreateICPMaps, Decay through the abstract ITMLib interfaces (synchronous, as DynSLAM calls them); "
                   f"{preroll}-frame pre-roll (decay queue live), {timed} timed frames, {repeats} repeats in a fresh process, median + "
                   "spread; stages_us = a separate pass with a device synchronise after every call; reference = unmodified CUDA engines, "
                   "nvcc sm_100a --use_fast_math")
    out["speedup_shim_vs_reference_cuda"] = out["speedup_median"]
    return out


# --------------------------------------------------------------------------------------------------
# roofline stress (BASELINE.json configs[4], SURVEY 8d config 5): 4 mm voxels, mu 16 mm — the same street at
# 12.5x finer voxels makes the visible list two orders of magnitude longer, so IntegrateIntoScene runs for
# hundreds of microseconds and its bandwidth fraction can be read without launch effects.
# --------------------------------------------------------------------------------------------------
def run_hires(local_rank, frames_n):
    """configs[4]: 4 mm voxels. frames_n <= 64: the short form of the default run (the stream's first frames, statistics over the
    second half). Longer: the stream at length — frames are generated and uploaded in chunks, the map grows to millions of blocks
    in a VBA sized for it, every IntegrateIntoScene launch is timed (CUDA events), decay off, no raycast."""
    import torch
    from dynslam_b200 import engine as E
    dev = torch.device("cuda", local_rank)
    W, H_ = synth.KITTI_W, synth.KITTI_H
    if frames_n > 64:
        return run_hires_long(local_rank, frames_n)
    nb, nbk, nex = 3000000, 0x400000, 0x100000
    frames = gen_frames_hires(5, frames_n)
    scene = E.Scene(E.SceneParams(voxelSize=0.004, mu=0.016, maxW=50), nb, nbk, nex, device=f"cuda:{local_rank}")
    eng = E.Engine(scene, (W, H_), decayRingItems=4 * nb)
    reco = E.SceneReconstructionEngine(eng)
    rs = E.VisualisationEngine(eng, scene).CreateRenderState((W, H_))
    reco.ResetScene(scene)
    views = [E.View(torch.from_numpy(f[0]).to(dev), torch.from_numpy(f[1]).to(dev), f[2], f[3]) for f in frames]
    torch.cuda.synchronize(dev)
    half = frames_n // 2
    for v in views[:half]:
        eng.process_frame_async(rs, v, None, None, decay=None, raycast=False)
    eng.sync(rs)
    b0 = eng.stats().totalIntegratedBlocks
    eng.set_timing(2)
    for v in views[half:]:
        eng.process_frame_async(rs, v, None, None, decay=None, raycast=False)
    eng.sync(rs)
    st = eng.stats()
    blocks, ms, n = st.totalIntegratedBlocks - b0, st.ring_ms_integrate, st.ring_count
    peak, _ = peaks()
    alg = blocks * BYTES_PER_BLOCK + n * W * H_ * 8
    out = {"workload": "4 mm voxels, mu 16 mm, depth clamp 8 m, same street (configs[4])", "frames": n,
           "visible_blocks": rs.noVisibleBlocks, "allocated_blocks": nb - 1 - scene.lastFreeBlockId,
           "mean_launch_us": 1000.0 * ms / max(n, 1), "achieved": alg / (ms / 1000.0) / 1e9 if ms > 0 else 0.0, "unit": "GB/s",
           "peak": peak, "mvoxels_per_s": blocks * 512 / (ms / 1000.0) / 1e6 if ms > 0 else 0.0}
    out["frac"] = out["achieved"] / peak
    eng.close()
    return out


# --------------------------------------------------------------------------------------------------
# view builder (SURVEY 8(f) rank 1): ITMViewBuilder::UpdateView of one raw KITTI-shaped frame through the real
# ITMLib classes — the reference's ITMViewBuilder_CUDA (7 launches) vs ITMViewBuilder_B200 (one fused kernel)
# --------------------------------------------------------------------------------------------------
def run_view_builder(frames, iters=60):
    from tests import harnesslib as HL
    if not HL.available():
        return {"error": "oracle/_ref/libitmharness.so not built"}
    raw = np.round(frames[0][0] * 1000.0).astype(np.int16)
    out = {"what": "UpdateView(rgb, raw int16 depth, useBilateralFilter=true) at 1242x375: 'update_view_us' = the call as "
                   "ITMMainEngine makes it (two blocking H2D copies from ITMLib's pinned host images + conversion + 5 filter passes "
                   "+ copy), 'device_only_us' = the same stages on a device-resident raw image; wall clock, device synchronised",
           "alg_bytes": raw.size * 6}
    for name, impl in (("reference_cuda_build", HL.REFERENCE_CUDA), ("b200", HL.B200_SHIM)):
        vb = HL.ViewBuilderHarness(impl, synth.KITTI_W, synth.KITTI_H, frames[0][3])
        vb.update_view(raw, frames[0][1])
        vb.time_update_view(5); vb.time_device_only(5)
        out[name] = {"update_view_us": 1000.0 * vb.time_update_view(iters), "device_only_us": 1000.0 * vb.time_device_only(iters)}
        vb.close()
    out["speedup_device_only"] = out["reference_cuda_build"]["device_only_us"] / out["b200"]["device_only_us"]
    return out


# --------------------------------------------------------------------------------------------------
# instance frame splitting + compositing (SURVEY 8(f) ranks 2-3): HBM-bound byte work, so each gets a roofline line.
# 7 cars (configs[2]) at 1242x375; L2 flushed before every timed launch; CUDA events on the engine's stream.
# --------------------------------------------------------------------------------------------------
def run_frames_ops(local_rank, iters=30, ncars=7):
    import torch
    from dynslam_b200 import engine as E
    dev = torch.device("cuda", local_rank)
    W, H_ = synth.KITTI_W, synth.KITTI_H
    stream = torch.cuda.Stream(device=dev)
    peak, _ = peaks()
    with torch.cuda.stream(stream):
        eng = E.Engine(E.Scene(E.SceneParams(), 2048, 0x800, 0x400, device=f"cuda:{local_rank}"), (W, H_), stream=stream.cuda_stream)
        fr = E.InstanceFrames(eng)
        rng = np.random.default_rng(7)
        rgb0 = torch.from_numpy(rng.integers(0, 256, (H_, W, 4), dtype=np.uint8)).to(dev)
        depth0 = torch.from_numpy(rng.uniform(0.5, 20.0, (H_, W)).astype(np.float32)).to(dev)
        ops, keep = [], []
        for i in range(ncars):           # car-sized boxes (~150x90 px) spread over the frame, elliptical silhouettes
            bw, bh = 150 + 10 * i, 90 + 4 * i
            x0, y0 = 40 + i * 160, 120 + (i % 3) * 40
            yy, xx = np.mgrid[0:bh, 0:bw]
            m = ((((xx - bw / 2) / (bw / 2)) ** 2 + ((yy - bh / 2) / (bh / 2)) ** 2) <= 1.0).astype(np.uint8)
            t = torch.from_numpy(m).to(dev)
            mask = E.make_mask((x0, y0, x0 + bw - 1, y0 + bh - 1), t)
            drgb = torch.zeros((H_, W, 4), dtype=torch.uint8, device=dev)
            ddep = torch.zeros((H_, W), dtype=torch.float32, device=dev)
            keep.append((t, mask, drgb, ddep))
            ops.append((E.EXTRACT, mask, mask, drgb, ddep))
        flush = torch.zeros(256 * 1024 * 1024 // 4, dtype=torch.int32, device=dev)
        rgb, depth = rgb0.clone(), depth0.clone()

        def timed(fn, reset, kernel):
            # Kernel time from the library's launch trace (an event pair right around the launch, b200_set_timing(3)); the
            # L2 flush is enqueued just before and nothing synchronises in between, so the launch never waits for the host.
            eng.set_timing(3)
            for it in range(iters + 3):
                reset()
                flush.add_(1)
                fn()
            stream.synchronize()
            d = [b - a for name, a, b in eng.trace() if name == kernel][3:]
            eng.set_timing(0)
            return sum(d) / len(d)

        def reset_split():
            rgb.copy_(rgb0); depth.copy_(depth0)
        us_split = timed(lambda: fr.ProcessSilhouettes(rgb, depth, ops, sync=False, wait_inputs=False), reset_split, "k_process_silhouettes")
        # algorithmic bytes: the frame is read once (8 B/px); every instance frame is written in full (8 B/px each, the
        # reference's two memsets + copies); the blanked pixels of the main frame are written back
        blanked = int((depth == 0).sum().item())
        bytes_split = W * H_ * 8 + ncars * W * H_ * 8 + blanked * 8
        layers = [(k[2], k[3], E.MATPLOTLIB2_PALETTE[i % 10]) for i, k in enumerate(keep)]
        out_c, out_d = rgb0.clone(), depth0.clone()

        def reset_cmp():
            out_c.copy_(rgb0); out_d.copy_(depth0)
        us_cmp = timed(lambda: fr.CompositeInstances(out_c, out_d, layers, dim_factor=0.10, tint_strength=1.0, wait_inputs=False), reset_cmp,
                       "k_composite_layers")
        # every layer's depth is read (4 B/px); its colour only where it wins; background read + written (16 B/px)
        bytes_cmp = W * H_ * 16 + ncars * W * H_ * 4
        # evaluation consumer (Evaluation::EvaluateDepth): 120 k LIDAR returns x the reference's 14 callbacks on a frame-sized depth
        evaluation = None
        try:
            fx, bl = 721.5377, 0.5371657
            cxp, cyp = W / 2.0 + 3.2, H_ / 2.0 - 5.1
            v2c = np.array([[7.5337e-03, -9.999714e-01, -6.16602e-04, -4.069766e-03], [1.480249e-02, 7.280733e-04, -9.998902e-01, -7.631618e-02],
                            [9.998621e-01, 7.523790e-03, 1.480755e-02, -2.717806e-01], [0.0, 0.0, 0.0, 1.0]])
            pl = np.array([[fx, 0, cxp, 44.85728], [0, fx, cyp, 0.2163791], [0, 0, 1, 2.745884e-03]])
            pr = pl.copy(); pr[0, 3] -= fx * bl
            npts = 120000
            z = rng.uniform(0.6, 40.0, npts); u = rng.uniform(-30, W + 30, npts); r_ = rng.uniform(-20, H_ + 20, npts)
            cam = np.stack([(u - cxp) * z / fx, (r_ - cyp) * z / fx, z, np.ones(npts)], 1)
            velo = (np.linalg.inv(v2c) @ cam.T).T
            pts = np.concatenate([velo[:, :3], rng.uniform(0, 1, (npts, 1))], 1).astype(np.float32)
            d_pts = torch.from_numpy(pts).to(dev)
            rendered = depth0.clone(); rendered[rendered > 18.0] = 0.0
            inp = torch.clamp(torch.round(depth0 * 1000.0 + 50.0), 0, 32000).to(torch.int16)
            ev = E.Evaluation(eng, v2c, pl, pr, bl, W, H_, 0.5, 30.0)
            res = None
            eng.set_timing(3)
            t_wall = []
            for it in range(iters + 3):
                flush.add_(1); stream.synchronize()
                t0 = time.perf_counter()
                res = ev.EvaluateDepth(d_pts, rendered, inp)
                t_wall.append((time.perf_counter() - t0) * 1e6)
            d = [b - a for name, a, b in eng.trace() if name == "k_evaluate_depth"][3:]
            eng.set_timing(0)
            evaluation = {"kernel_us": sum(d) / len(d), "call_us": float(np.median(t_wall[3:])), "points": npts, "callbacks": 14,
                          "measurements": res[0][0]["measurement_count"], "alg_bytes": npts * 16 + res[0][0]["measurement_count"] * 6,
                          "what": "b200_evaluate_depth: every LIDAR return of a frame through the reference's 14 callbacks, one launch; call_us = the synchronous call incl. the counter read-back"}
        except Exception as ex:
            evaluation = {"error": str(ex)}
        eng.close()
    return {"evaluation": evaluation,
            "instance_split": {"us": us_split, "ops": ncars, "alg_bytes": bytes_split, "achieved": bytes_split / us_split / 1e3,
                               "peak": peak, "unit": "GB/s", "frac": bytes_split / us_split / 1e3 / peak,
                               "what": "b200_process_silhouettes_async: 7 detections cut out of a 1242x375 frame into 7 instance frames, one launch"},
            "composite": {"us": us_cmp, "layers": ncars, "alg_bytes": bytes_cmp, "achieved": bytes_cmp / us_cmp / 1e3, "peak": peak,
                          "unit": "GB/s", "frac": bytes_cmp / us_cmp / 1e3 / peak,
                          "what": "b200_composite_instances (synchronous call): background dim + 7 layers z-composited, one launch"}}


# --------------------------------------------------------------------------------------------------
# configs[3] (SURVEY 8d config 4): Decay(forceAllVoxels) — FullDecay, Reco_CUDA.cu:430-475 — over a volume pre-filled to
# `blocks` allocated hash blocks (2 M at 1 GPU, 250 k per GPU at 8), table enlarged to 0x400000 buckets; voxel weights drawn so
# that 30 % of the voxels of a surviving block are noise (w_depth <= maxWeight) and 10 % of the blocks become empty and are
# deleted. Mblocks/s and the fraction of the HBM roofline at 4116 B per examined block + 8 B per reset voxel (SURVEY 8d).
# --------------------------------------------------------------------------------------------------
def run_decay_sweep(local_rank, blocks, repeats=3):
    import torch
    from dynslam_b200 import abi, engine as E
    dev = torch.device("cuda", local_rank)
    nbk, nex = 0x400000, 0x100000
    ent, alloc_list, excess_list, last_free, last_free_ex = synth.prefilled_hash(blocks, nbk, nex, seed=4)
    scene = E.Scene(E.SceneParams(), blocks, nbk, nex, device=f"cuda:{local_rank}")
    eng = E.Engine(scene, (64, 48))
    reco = E.SceneReconstructionEngine(eng)
    rs = E.VisualisationEngine(eng, scene).CreateRenderState((64, 48))
    reco.ResetScene(scene)
    h_ent = torch.from_numpy(ent.view(np.uint8).reshape(-1))
    gen = torch.Generator(device=dev); gen.manual_seed(4)
    empty_block = torch.rand(blocks, generator=gen, device=dev) < 0.10          # every voxel of these is noise -> block deleted
    times, freed_all, reset_all = [], [], []
    for rep in range(repeats + 1):                                               # pass 0 is the warm-up
        scene.hash.copy_(h_ent.to(dev))
        scene.allocationList.copy_(torch.from_numpy(alloc_list).to(dev))
        scene.excessList.copy_(torch.from_numpy(excess_list).to(dev))
        vox = scene.voxels.view(blocks, 512, 8)
        chunk = 1 << 16
        n_reset = 0
        for b0 in range(0, blocks, chunk):
            b1 = min(blocks, b0 + chunk)
            w = torch.randint(2, 51, (b1 - b0, 512), generator=gen, device=dev, dtype=torch.int16)
            noise = torch.rand((b1 - b0, 512), generator=gen, device=dev) < 0.30
            w = torch.where(noise | empty_block[b0:b1, None], torch.ones_like(w), w)
            n_reset += int((w == 1).sum().item())
            v = vox[b0:b1]
            v[..., 0:2] = torch.randint(0, 256, (b1 - b0, 512, 2), generator=gen, device=dev, dtype=torch.uint8)
            v[..., 2] = w.to(torch.uint8)
            v[..., 3:7] = 7
            v[..., 7] = 0
        scene.c.lastFreeBlockId, scene.c.lastFreeExcessListId = last_free, last_free_ex
        torch.cuda.synchronize(dev)
        before = reco.GetDecayedBlockCount()
        t0 = time.perf_counter()
        reco.Decay(scene, rs, 1, 0, True)            # synchronous C-ABI call: returns with the counters on the host
        dt = time.perf_counter() - t0
        if rep > 0:
            times.append(dt); freed_all.append(reco.GetDecayedBlockCount() - before); reset_all.append(n_reset)
    expected_freed = int(empty_block.sum().item())
    st_ptr = scene.hash.view(-1, 20)[:, 12:16].contiguous().view(torch.int32).view(-1)
    still = int((st_ptr >= 0).sum().item())
    t = float(np.median(times))
    alg = blocks * 4116 + reset_all[-1] * 8
    peak, _ = peaks()
    out = {"workload": f"Decay(maxWeight 1, minAge 0, forceAllVoxels) over {blocks} allocated blocks, 0x400000 buckets (configs[3])",
           "blocks": blocks, "ms": 1000.0 * t, "passes_ms": [1000.0 * x for x in times], "mblocks_per_s": blocks / t / 1e6,
           "freed_blocks": int(freed_all[-1]), "expected_freed": expected_freed, "still_allocated": still,
           "conservation_ok": bool(freed_all[-1] == expected_freed and still + freed_all[-1] == blocks and scene.lastFreeBlockId == freed_all[-1] - 1),
           "reset_voxels": int(reset_all[-1]), "alg_bytes": int(alg), "achieved": alg / t / 1e9, "peak": peak, "unit": "GB/s",
           "frac": alg / t / 1e9 / peak, "timing": "wall clock around the synchronous b200_decay call (includes its counter round trip)"}
    eng.close()
    return out


def _hires_chunk(args):
    seed, first, count, length_m = args
    scene = synth.StreetScene(seed=seed, length_m=length_m)
    return [synth.kitti_frame(scene, f, zmax=8.0) for f in range(first, first + count)]


def gen_frames_hires(seed, count, first=0, length_m=60.0, workers=1):
    if workers <= 1 or count < 8:
        return _hires_chunk((seed, first, count, length_m))
    import multiprocessing as mp
    per = (count + workers - 1) // workers
    jobs = [(seed, first + i * per, min(per, count - i * per), length_m) for i in range(workers) if i * per < count]
    with mp.get_context("fork").Pool(len(jobs)) as pool:
        parts = pool.map(_hires_chunk, jobs)
    return [f for p in parts for f in p]


def run_hires_long(local_rank, frames_n, chunk=100):
    import torch
    from dynslam_b200 import engine as E
    dev = torch.device("cuda", local_rank)
    W, H_ = synth.KITTI_W, synth.KITTI_H
    length_m = frames_n * 0.8 + 60.0
    # the 4 mm map of this street gains ~11 k blocks per frame (0.8 m of new street): size the VBA for the whole stream
    per_frame = 11500
    nb = min(int(160e9 // 4096), int(260000 + per_frame * frames_n * 1.15))
    nbk, nex = 0x2000000, 0x800000
    scene = E.Scene(E.SceneParams(voxelSize=0.004, mu=0.016, maxW=50), nb, nbk, nex, device=f"cuda:{local_rank}")
    eng = E.Engine(scene, (W, H_), decayRingItems=4 * 65536)
    reco = E.SceneReconstructionEngine(eng)
    rs = E.VisualisationEngine(eng, scene).CreateRenderState((W, H_))
    reco.ResetScene(scene)
    done, blocks, ms, launches, stopped = 0, 0, 0.0, 0, None
    workers = max(1, min(32, (os.cpu_count() or 2) - 2))
    t_all = time.perf_counter()
    while done < frames_n:
        n = min(chunk, frames_n - done)
        frames = gen_frames_hires(5, n, first=done, length_m=length_m, workers=workers)
        views = [E.View(torch.from_numpy(f[0]).to(dev), torch.from_numpy(f[1]).to(dev), f[2], f[3]) for f in frames]
        torch.cuda.synchronize(dev)
        b0 = eng.stats().totalIntegratedBlocks
        eng.set_timing(2)
        try:
            for v in views:
                eng.process_frame_async(rs, v, None, None, decay=None, raycast=False)
            eng.sync(rs)
        except RuntimeError as ex:          # VBA / excess list exhausted: report how far the stream got
            stopped = str(ex)
            break
        st = eng.stats()
        if done >= 100 or frames_n <= 100:   # the first 100 frames build the near field; statistics from then on
            blocks += st.totalIntegratedBlocks - b0; ms += st.ring_ms_integrate; launches += st.ring_count
        eng.set_timing(0)
        done += n
    peak, _ = peaks()
    alg = blocks * BYTES_PER_BLOCK + launches * W * H_ * 8
    out = {"workload": f"4 mm voxels, mu 16 mm, depth clamp 8 m, same street, {frames_n}-frame stream (configs[4])", "frames_requested": frames_n,
           "frames_done": done, "frames_timed": launches, "stopped": stopped, "vba_blocks": nb, "vba_gb": nb * 4096 / 1e9,
           "visible_blocks": rs.noVisibleBlocks, "allocated_blocks": nb - 1 - scene.lastFreeBlockId,
           "mean_launch_us": 1000.0 * ms / max(launches, 1), "achieved": alg / (ms / 1000.0) / 1e9 if ms > 0 else 0.0, "unit": "GB/s",
           "peak": peak, "mvoxels_per_s": blocks * 512 / (ms / 1000.0) / 1e6 if ms > 0 else 0.0, "wall_s": time.perf_counter() - t_all}
    out["frac"] = out["achieved"] / peak
    eng.close()
    return out


# --------------------------------------------------------------------------------------------------
# own arm
# --------------------------------------------------------------------------------------------------
def run_own(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from dynslam_b200 import abi, engine as E

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W, H_ = synth.KITTI_W, synth.KITTI_H
    K, Wm = args.steps, args.warmup
    n_e2e = args.e2e_steps
    n_raw = args.e2e_raw_steps if world == 1 else 0
    total_frames = args.preroll + Wm + K + 3 + n_e2e + n_raw
    length_m = total_frames * 0.8 + 60.0
    # N = 1: configs[1], the static map alone. N > 1: configs[2] — ONE street, N - 1 cars; rank 0 owns the static map (cars cut
    # out of its frames), rank r > 0 owns car r - 1's volume (InstanceReconstructor.cpp:363-389: mu 1.0, voxel 0.035, 7142 blocks)
    ncars = world - 1
    t_gen = time.perf_counter()
    workers = max(1, min(16, (os.cpu_count() or 2) // max(world, 1)))
    if world == 1:
        frames = gen_frames_parallel(6, 0, total_frames, length_m, workers)
    else:
        frames = gen_frames_cars_parallel(6, 0, total_frames, length_m, ncars, workers)
        if rank > 0:
            car = synth.FollowedCar(rank - 1, seed=3)
    log(f"[rank {rank}] generated {len(frames)} frames in {time.perf_counter() - t_gen:.1f}s")

    def host_pose(i):
        M = frames[i][2]
        return M if (world == 1 or rank == 0) else car.object_pose(i, M)

    def host_frame(i):
        """the host-side frame of THIS rank's volume (e2e phases): rank 0 the street frame, rank r the frame masked to its car"""
        depth, rgb, M, proj = frames[i][:4]
        if world == 1 or rank == 0:
            return depth, rgb, M
        m = frames[i][4][rank - 1]
        full = np.zeros(depth.shape, dtype=bool)
        if m is not None:
            (x0, y0, x1, y1), data = m
            full[y0:y1 + 1, x0:x1 + 1] = data.astype(bool)
        return (np.where(full, depth, np.float32(0.0)).astype(np.float32), np.where(full[..., None], rgb, np.uint8(255)).astype(np.uint8),
                car.object_pose(i, M))

    # Host buffers of the e2e phases are pinned NOW, long before they are used: pinning several hundred MB was followed, some
    # milliseconds later, by a one-off 50-70 ms host stall (seen as a single gap between two pipelined submissions, with the
    # clock sampler paused and the GC off), which a 50 ms e2e phase cannot absorb.
    e2e_first = args.preroll + Wm + K + 3
    h_depth = [torch.from_numpy(host_frame(e2e_first + i)[0]).pin_memory() for i in range(n_e2e)]
    h_rgb = [torch.from_numpy(host_frame(e2e_first + i)[1]).pin_memory() for i in range(n_e2e)]
    h_raw = [torch.from_numpy(np.round(frames[e2e_first + n_e2e + i][0] * 1000.0).astype(np.int16)).pin_memory() for i in range(n_raw)]
    h_rgb2 = [torch.from_numpy(frames[e2e_first + n_e2e + i][1]).pin_memory() for i in range(n_raw)]
    h_out = [torch.zeros(H_ * W * 4, dtype=torch.uint8).pin_memory() for _ in range(2)]

    stream = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(stream):
        instance = world > 1 and rank > 0
        if instance:   # per-car volume: InstanceReconstructor.cpp:365-389 (mu 1.0, voxel 0.035, 5*5*10 m / 0.035 -> 7142 blocks), full-size table
            scene = E.Scene(E.SceneParams(voxelSize=0.035, mu=1.0, maxW=50), 7142, NUM_BUCKETS, EXCESS, device=f"cuda:{local_rank}")
        else:
            scene = E.Scene(E.SceneParams(), NUM_BLOCKS, NUM_BUCKETS, EXCESS, device=f"cuda:{local_rank}")
        eng = E.Engine(scene, (W, H_), stream=stream.cuda_stream)
        reco = E.SceneReconstructionEngine(eng)
        vis = E.VisualisationEngine(eng, scene)
        rs = vis.CreateRenderState((W, H_))
        reco.ResetScene(scene)
        points = torch.zeros(H_ * W * 4, dtype=torch.float32, device=dev)
        normals = torch.zeros(H_ * W * 4, dtype=torch.float32, device=dev)
        # multi-volume exchange (csrc/comm.cu): two slots of this volume's colour + depth render, rank 0 also of the composite
        xch, frames_api = None, None
        if world > 1:
            from dynslam_b200 import multi
            xch = multi.VolumeExchange(eng, (W, H_), rank, world)
            frames_api = E.InstanceFrames(eng)
            lay_col = [torch.zeros((H_, W, 4), dtype=torch.uint8, device=dev) for _ in range(2)]
            lay_dep = [torch.zeros((H_, W), dtype=torch.float32, device=dev) for _ in range(2)]
            out_col = [torch.zeros((H_, W, 4), dtype=torch.uint8, device=dev) for _ in range(2)] if rank == 0 else [None, None]
            out_dep = [torch.zeros((H_, W), dtype=torch.float32, device=dev) for _ in range(2)] if rank == 0 else [None, None]
            inst_rgb = torch.zeros((H_, W, 4), dtype=torch.uint8, device=dev)
            inst_depth = torch.zeros((H_, W), dtype=torch.float32, device=dev)
        flush_buf = torch.zeros(256 * 1024 * 1024 // 4, dtype=torch.int32, device=dev) if args.flush_l2 else None   # 2x the 126 MB L2

        frame_no = [0]

        def dev_view(fr):
            """device-resident inputs of one step: the frame, and at N > 1 the silhouette masks this rank needs"""
            depth, rgb, M, proj = fr[:4]
            d = torch.from_numpy(depth).to(dev, non_blocking=False)
            c = torch.from_numpy(rgb).to(dev, non_blocking=False)
            if world == 1:
                return E.View(d, c, M, proj)
            masks = fr[4]
            f = frame_no[0]; frame_no[0] += 1
            if rank == 0:      # RemoveSilhouette for every visible car (InstanceReconstructor.cpp:226-285: delete_mask)
                ops, keep = [], []
                for m in masks:
                    if m is not None:
                        t = torch.from_numpy(m[1]).to(dev)
                        keep.append(t)
                        ops.append((E.REMOVE, None, E.make_mask(m[0], t), None, None))
                v = E.View(d, c, M, proj)
                v.ops, v.keep = (E.InstanceFrames.prepare_ops(ops) if ops else None), keep
                return v
            m = masks[rank - 1]  # ProcessSilhouette: the car's pixels are copied into the instance frame (:91-127), fused with the object pose
            v = E.View(inst_depth, inst_rgb, car.object_pose(f, M), proj)
            v.src = (d, c)
            if m is not None:
                t = torch.from_numpy(m[1]).to(dev)
                mk = E.make_mask(m[0], t)
                v.ops, v.keep = E.InstanceFrames.prepare_ops([(E.EXTRACT, mk, mk, inst_rgb, inst_depth)]), [t]
            else:
                v.ops, v.keep = None, []
            return v

        step_no = [0]
        diag = os.environ.get("B200_BENCH_DIAG", "")

        def step(view, host=None):
            """one frame of this rank's volume; at N > 1 preceded by the instance split and followed by the hand-over of the
            volume's colour + depth render to rank 0 (composited there), all enqueued without host synchronisation"""
            if world == 1:
                eng.process_frame_async(rs, view, points, normals, decay=DECAY)
                return
            k = step_no[0]; step_no[0] += 1
            s = k & 1
            # B200_BENCH_DIAG (measurement aid, not a bench mode): noxch = no hand-over / composite, nosplit = no silhouette pass,
            # norender = no extra colour / depth renders — to attribute the per-step cost of configs[2] over configs[1]
            do_xch, do_split, do_render = "noxch" not in diag, "nosplit" not in diag, "norender" not in diag
            if do_xch and "norelease" not in diag:
                xch.release(k)                               # slot s was handed over with frame k - 2: its buffers are free again
            if rank == 0:
                if view.ops and do_split:
                    frames_api.ProcessSilhouettes(view.rgb, view.depth, view.ops, sync=False, wait_inputs=False)
                rs.c.d_raycastImage = lay_col[s].data_ptr()   # the static map's layer is its shaded raycast image (the ICP pass writes it)
                eng.process_frame_async(rs, view, points, normals, decay=DECAY, depth_out=lay_dep[s] if do_render else None)
                if do_xch:
                    xch.submit(k, lay_col[s], lay_dep[s], out_col[s], out_dep[s])
            else:
                if view.ops and do_split:
                    frames_api.ProcessSilhouettes(view.src[1], view.src[0], view.ops, sync=False, wait_inputs=False)
                elif do_split:                                # car not in view: the reference feeds nothing; an empty frame is the no-op
                    inst_depth.zero_()
                eng.process_frame_async(rs, view, points, normals, decay=DECAY, colour_out=lay_col[s] if do_render else None,
                                        depth_out=lay_dep[s] if do_render else None)
                if do_xch:
                    xch.submit(k, lay_col[s], lay_dep[s])

        sampler = ClockSampler(local_rank)
        if "nosampler" not in diag:
            sampler.start()
        import gc
        gc.collect()
        gc.disable()        # no collector pauses inside the timed loops (they show up as millisecond gaps between two frame submissions)
        # ---- pre-roll: build the map to steady state (untimed set-up) ----
        idx = 0
        for _ in range(args.preroll):
            step(dev_view(frames[idx])); idx += 1
        eng.sync(rs)
        views = [dev_view(frames[idx + i]) for i in range(Wm + K + 3)]
        idx += Wm + K + 3
        for i in range(Wm):
            step(views[i])
        eng.sync(rs)
        launches0 = eng.stats().launches
        blocks0 = eng.stats().totalIntegratedBlocks
        eng.set_timing(2)
        clk_first = len(sampler.rows)
        if world > 1:
            xch.finish()           # nothing of the pre-roll's exchange is in flight when the ranks line up
            dist.barrier()
        torch.cuda.synchronize(dev)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        flush_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)] if args.flush_l2 else []
        t0 = time.perf_counter()
        ev0.record(stream)
        for i in range(K):
            if args.flush_l2:       # evict L2 between timed iterations; the flush itself is timed and subtracted
                flush_ev[i][0].record(stream)
                flush_buf.add_(1)
                flush_ev[i][1].record(stream)
            if args.profile_step == i:   # ncu --profile-from-start off: exactly this frame's kernels are captured
                torch.cuda.synchronize(dev)
                torch.cuda.cudart().cudaProfilerStart()
            step(views[Wm + i])
            if args.profile_step == i:
                torch.cuda.synchronize(dev)
                torch.cuda.cudart().cudaProfilerStop()
        if world > 1:      # the last two hand-overs (and rank 0's composites) belong to the timed region
            xch.release(step_no[0]); xch.release(step_no[0] + 1)
        ev1.record(stream)
        torch.cuda.synchronize(dev)
        if world > 1:
            xch.finish()
            dist.barrier()
        wall_ms = (time.perf_counter() - t0) * 1000.0
        flush_ms = sum(a.elapsed_time(b) for a, b in flush_ev)
        gpu_ms = ev0.elapsed_time(ev1) - flush_ms
        wall_ms -= flush_ms
        eng.sync(rs)
        st = eng.stats()
        time.sleep(0.05)
        sampler.pause(True)
        clk_timed_end = len(sampler.rows)      # the sampler process stays alive (paused) through the e2e phases: terminating nvidia-smi stalls
                                               # the driver for tens of milliseconds, which used to land in the e2e timing
        launches = st.launches - launches0
        blocks = st.totalIntegratedBlocks - blocks0
        int_ms, int_n = st.ring_ms_integrate, st.ring_count
        n_vis = rs.noVisibleBlocks
        # sanity of the timed work: the last timed frame's raycast must have hit the surface on a large part of the image
        # (a broken expected-depth image makes every ray exit at once and the frame look fast)
        rays_hit = int((rs.raycastResult.view(-1, 4)[:, 3] > 0).sum().item())
        if (not instance) and (rays_hit < 0.3 * W * H_ or n_vis < 1000):
            raise RuntimeError(f"bench sanity check failed: {rays_hit} of {W * H_} rays hit the surface, {n_vis} visible blocks")
        used_blocks = scene.numBlocks - 1 - scene.lastFreeBlockId
        decayed = reco.GetDecayedBlockCount()
        snap = gpu_snapshot(scene, rs, points) if (rank == 0 and world == 1 and args.parity_check) else None   # the state the timed steps left behind
        if world > 1 and rank == 0:     # sanity of the exchange: the composite of the last timed frame carries pixels of every visible car
            comp_d, own_d = out_dep[(step_no[0] - 1) & 1], lay_dep[(step_no[0] - 1) & 1]
            closer = int(((comp_d != own_d)).sum().item())
            log(f"[rank 0] composite: {closer} pixels taken from instance layers")
        if args.dump_outputs and rank == 0:
            # what the last timed step handed its caller, before the untimed frames below overwrite it: ICP points and normals,
            # ray points and the shaded image of rank 0's volume; at N > 1 rank 0's composite instead of its own image
            out = {"points": points.view(H_, W, 4), "normals": normals.view(H_, W, 4), "raycast_result": rs.raycastResult.view(H_, W, 4)}
            if world == 1:
                out["raycast_image"] = rs.raycastImage.view(H_, W, 4)
            else:
                out["composite_colour"], out["composite_depth"] = out_col[(step_no[0] - 1) & 1], out_dep[(step_no[0] - 1) & 1]
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, t in out.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), t.float().cpu().numpy())
            log(f"[rank 0] wrote {', '.join(out)} of timed step {K - 1} to {args.dump_outputs}")
        # per-stage breakdown of a few extra frames (per-frame sync; not part of the timed region)
        eng.set_timing(1)
        stage = np.zeros(6)
        for i in range(3):
            step(views[Wm + K + i])
            eng.sync(rs)
            s = eng.stats()
            stage += np.array([s.ms_allocate, s.ms_integrate, s.ms_expected, s.ms_raycast, s.ms_decay, s.ms_total])
        stage /= 3.0
        eng.set_timing(0)

        # ---- e2e: host buffers -> H2D -> frame -> D2H image, every step ----
        assert idx == e2e_first, (idx, e2e_first)
        ev = E.View(torch.zeros((H_, W), dtype=torch.float32, device=dev), torch.zeros((H_, W, 4), dtype=torch.uint8, device=dev),
                    frames[idx][2], frames[idx][3])
        e2e_warm = min(3, n_e2e // 2)
        e2e_marks = []
        t_e2e = 0.0
        for i in range(n_e2e):
            if i == e2e_warm:
                eng.host_frame_wait(0); eng.host_frame_wait(1)
                torch.cuda.synchronize(dev)
                if world > 1:
                    xch.finish()
                    dist.barrier()
                t_e2e = time.perf_counter()
            slot = i & 1
            eng.host_frame_wait(slot)          # frame i-2 (same staging slot) has delivered its image
            e2e_marks.append(time.perf_counter())
            ev.set_pose(host_pose(idx + i))
            # public API: host depth+RGB in, grey raycast image out; copies of neighbouring frames overlap the kernels
            if world > 1:
                k = step_no[0]; step_no[0] += 1
                xch.release(k)
                rs.c.d_raycastImage = lay_col[k & 1].data_ptr()       # every volume hands over its shaded raycast image + depth render
                eng.host_frame_submit(rs, ev, h_depth[i], h_rgb[i], points, normals, decay=DECAY, h_out=h_out[slot], slot=slot,
                                      depth_out=lay_dep[k & 1])
                xch.submit(k, lay_col[k & 1], lay_dep[k & 1], out_col[k & 1], out_dep[k & 1])
            else:
                eng.host_frame_submit(rs, ev, h_depth[i], h_rgb[i], points, normals, decay=DECAY, h_out=h_out[slot], slot=slot)
        eng.host_frame_wait(0); eng.host_frame_wait(1)
        if world > 1:
            xch.finish()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        t_e2e = time.perf_counter() - t_e2e
        e2e_frames = n_e2e - e2e_warm

        # ---- e2e from RAW sensor frames: int16 depth + RGB in, UpdateView (conversion + 5-pass bilateral filter) on the
        # device, fused frame, grey image out (what DynSLAM does per frame from InfiniTamDriver::UpdateView onwards) ----
        e2e_raw = None
        if n_raw > 3:
            calib = E.make_view_calib()
            base = idx + n_e2e
            t_raw = 0.0
            raw_marks = []
            for i in range(n_raw):
                if i == 3:
                    eng.host_frame_wait(0); eng.host_frame_wait(1)
                    torch.cuda.synchronize(dev)
                    t_raw = time.perf_counter()
                slot = i & 1
                eng.host_frame_wait(slot)
                raw_marks.append(time.perf_counter())
                ev.set_pose(frames[base + i][2])
                eng.host_frame_submit_raw(rs, ev, h_raw[i], h_rgb2[i], calib, points, normals, decay=DECAY, h_out=h_out[slot], slot=slot)
            eng.host_frame_wait(0); eng.host_frame_wait(1)
            torch.cuda.synchronize(dev)
            t_raw = time.perf_counter() - t_raw
            e2e_raw = {"frame_ms": frame_gaps(raw_marks[3:]), "value": (n_raw - 3) / t_raw, "unit": "frames/s", "h2d_bytes_per_step": W * H_ * 6, "d2h_bytes_per_step": W * H_ * 4,
                       "steps": n_raw - 3, "what": "raw int16 depth + RGB in -> UpdateView with bilateral filter -> fused frame -> image out"}

        # ---- meshing of the map the run built (SURVEY 8(f) rank 4; untimed region, 1 GPU only) ----
        meshing = None
        if world == 1 and args.harness_frames > 0:
            try:
                mesh = E.Mesh(scene)        # ITMMesh: noMaxTriangles = SDF_LOCAL_BLOCK_NUM * 32
                me = E.MeshingEngine(eng)
                ts = []
                for _ in range(3):
                    torch.cuda.synchronize(dev)
                    t0 = time.perf_counter()
                    ntri = me.MeshScene(mesh, scene)
                    ts.append((time.perf_counter() - t0) * 1e3)
                allocated = scene.numBlocks - 1 - scene.lastFreeBlockId
                meshing = {"ms": sorted(ts)[1], "passes_ms": ts, "triangles": int(ntri), "allocated_blocks": int(allocated),
                           "mblocks_per_s": allocated / (sorted(ts)[1] / 1e3) / 1e6,
                           "what": "b200_mesh_scene (synchronous, incl. its counter round trip) over the map the timed run built; triangles in the CPU engine's order"}
                del mesh
            except Exception as ex:
                meshing = {"error": str(ex)}

    gc.enable()
    sampler.stop()
    clk_all = len(sampler.rows)
    sampler.rows = sampler.rows[max(clk_first - 1, 0):clk_timed_end] or sampler.rows   # samples taken during the timed region
    clocks = sampler.summary()
    clocks["samples_since_start"] = clk_all

    decay_sweep = None
    if args.decay_blocks > 0:
        try:
            # configs[3]: 2 M blocks on one GPU; at N GPUs every rank sweeps its own share (2 M / N) concurrently
            torch.cuda.synchronize(dev)
            if world > 1:
                dist.barrier()
            ds = run_decay_sweep(local_rank, max(args.decay_blocks // world, 1024))
            if world > 1:
                t = torch.tensor([ds["ms"], float(ds["blocks"]), float(ds["alg_bytes"]), 1.0 if ds["conservation_ok"] else 0.0], dtype=torch.float64, device=dev)
                tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
                tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
                ds = dict(ds, ms=float(tmax[0]), blocks=int(tsum[1]), mblocks_per_s=float(tsum[1]) / (float(tmax[0]) / 1000.0) / 1e6,
                          achieved=float(tsum[2]) / (float(tmax[0]) / 1000.0) / 1e9 / world, alg_bytes=int(tsum[2]),
                          conservation_ok=bool(float(tsum[3]) == world), ranks=world,
                          note="max time over ranks, blocks summed; `achieved` is per GPU")
                ds["frac"] = ds["achieved"] / ds["peak"]
            decay_sweep = ds
        except Exception as ex:
            decay_sweep = {"error": str(ex)}


    # ---- reduce over ranks (max time) ----
    ms = max(gpu_ms, 0.0)
    if world > 1:
        # The ranks run in lock step (a volume may be at most two frames ahead of the compositor), so every rank's timed region
        # lasts as long as the slowest rank's INCLUDING that rank's L2 flushes, and the flushes take different times on different
        # ranks (84 us on a GPU that then waits, 128 us on the one that is busy). Subtracting each rank's OWN flush time before the
        # max would book the waiting for the slowest rank's longer flushes as work of the faster one (measured: 222 us "for" the
        # instance volume against 180 us for the static map that actually paces the job). So: max over ranks of the whole region,
        # minus the max over ranks of the flush time — the flushes on the critical path.
        log(f"[rank {rank}] own timed region: {gpu_ms / K * 1000.0:.1f} us/step on the device after {flush_ms / K * 1000.0:.1f} us/step of L2 flush")
        t = torch.tensor([gpu_ms + flush_ms, flush_ms, wall_ms + flush_ms, t_e2e, float(blocks), float(launches)], dtype=torch.float64, device=dev)
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms, wall_ms, t_e2e = float(tmax[0] - tmax[1]), float(tmax[2] - tmax[1]), float(tmax[3])
        blocks_all, launches_all = float(tsum[4]), float(tsum[5])
    else:
        blocks_all, launches_all = float(blocks), float(launches)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    fps = world * K / (ms / 1000.0)
    mvox = blocks_all * 512 / (ms / 1000.0) / 1e6
    peak, peak_src = peaks()
    alg_bytes = blocks * BYTES_PER_BLOCK + int_n * W * H_ * 8
    achieved = alg_bytes / (int_ms / 1000.0) / 1e9 if int_ms > 0 else 0.0
    footprint_mb = (n_vis * 4096 * 2 + (NUM_BUCKETS + EXCESS) * 21 + W * H_ * (8 + 8 + 16 + 4 + 32)) / 1e6

    parity = {"parity_checked": False, "why": "--no-parity-check"}
    if snap is not None:
        try:
            parity = parity_check(frames, args.preroll + Wm + K, snap)
            parity["decayed_blocks_gpu"] = int(decayed)
        except Exception as ex:
            parity = {"parity_checked": False, "why": f"oracle replay failed: {ex}"}
        snap = None

    cpu = None
    if args.cpu_steps > 0 and world == 1:      # the CPU baseline is timed at N = 1 only
        try:
            c = cpu_run(6, args.preroll, 1, args.cpu_steps, passes=1)
            cpu = {"value": c["fps"], "unit": "frames/s", "cores": c["cores"], "kind": "port",
                   "sample": f"{c['frames']} frames after the same {c['preroll']}-frame pre-roll of the same stream (decay queue live), "
                             f"fixed at {c['cores']} OpenMP threads; {c['mvoxels_per_s']:.1f} Mvoxels/s",
                   "ms_per_step": c["ms_per_step"]}
        except Exception as ex:  # the baseline is reported, never required for the GPU numbers
            cpu = {"value": None, "unit": "frames/s", "cores": 0, "kind": "port", "sample": f"failed: {ex}"}

    itm = None
    if world == 1 and args.harness_frames > 0:
        try:
            itm = run_itm_harness(args.preroll, args.harness_frames)
        except Exception as ex:
            itm = {"error": str(ex)}

    hires = None
    if world == 1 and args.hires_frames > 0:
        try:
            hires = run_hires(local_rank, args.hires_frames)
        except Exception as ex:
            hires = {"error": str(ex)}

    vbuild = None
    if world == 1 and args.harness_frames > 0:
        try:
            vbuild = run_view_builder(frames)
        except Exception as ex:
            vbuild = {"error": str(ex)}

    frames_ops = None
    if world == 1 and args.harness_frames > 0:
        try:
            frames_ops = run_frames_ops(local_rank)
        except Exception as ex:
            frames_ops = {"error": str(ex)}

    line = {
        "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": dict(base_config(args.preroll),
                   l2=(f"explicit flush between timed steps (256 MB read-modify-write, timed with CUDA events and subtracted, "
                          f"{flush_ms / max(K, 1) * 1000:.0f} us each" + ("; N > 1: the ranks run in lock step, so the whole region is max-reduced and the "
                          "slowest rank's flushes are subtracted" if world > 1 else "") + f"); per-step footprint ~{footprint_mb:.0f} MB") if args.flush_l2 else
                         f"no flush (--no-flush-l2): per-step footprint ~{footprint_mb:.0f} MB, consecutive frames reuse L2",
                   integrate_impl=os.environ.get("B200_INTEGRATE_IMPL", "v4"),
                   parallelism=(f"configs[2]: one volume per GPU — rank 0 the static map (cars cut out with b200_process_silhouettes), ranks 1..{world - 1} one "
                                "car volume each (voxel 0.035, mu 1.0, 7142 blocks) fed by b200_process_silhouettes; every frame each rank's colour + "
                                "depth render goes to rank 0 (C++ exchange: copy-engine push over NVLink into rank 0's IPC-exported buffers, stream "
                                "memory operations for the flags, own stream + own host thread, two slots; NCCL for the bootstrap) and is composited "
                                "there inside the timed loop; value = volume-frames/s") if world > 1 else "1 volume"),
        "parity_checked": bool(parity.get("parity_checked")), "parity": parity,
        "mvoxels_per_s": mvox, "rays_hit": rays_hit, "visible_blocks": n_vis, "allocated_blocks": used_blocks, "decayed_blocks": int(decayed),
        "wall_ms_per_step": wall_ms / K,
        "stage_ms": {"allocate": stage[0], "integrate": stage[1], "expected_depths": stage[2], "raycast_icp": stage[3],
                     "decay": stage[4], "total": stage[5]},
        "roofline": {"kernel": "k_integrate_" + os.environ.get("B200_INTEGRATE_IMPL", "v4"), "bound": "hbm", "achieved": achieved,
                     "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None, "traffic": ncu_traffic(),
                     "peak_source": peak_src, "launches_timed": int_n, "mean_launch_us": 1000.0 * int_ms / max(int_n, 1),
                     "alg_bytes_per_launch": alg_bytes / max(int_n, 1)},
        "roofline_hires": hires,
        "decay_sweep": decay_sweep,
        "cpu_baseline": cpu,
        "itmlib_harness": itm,
        "view_builder": vbuild,
        "frames_ops": frames_ops,
        "e2e_raw": e2e_raw,
        "meshing": meshing,
        "e2e": {"value": world * e2e_frames / t_e2e, "unit": "frames/s", "h2d_bytes_per_step": W * H_ * 8,
                "d2h_bytes_per_step": W * H_ * 4, "steps": e2e_frames, "frame_ms": frame_gaps(e2e_marks[e2e_warm:])},
        "gpu_launches": int(launches_all),
        "clocks": clocks,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--preroll", type=int, default=230, help="untimed frames that build the map (> decay minAge)")
    ap.add_argument("--e2e-steps", type=int, default=203)
    ap.add_argument("--e2e-raw-steps", type=int, default=103, help="frames of the raw-sensor-frame e2e variant (1 GPU only)")
    ap.add_argument("--flush-l2", dest="flush_l2", action="store_true", default=True)
    ap.add_argument("--no-flush-l2", dest="flush_l2", action="store_false")
    ap.add_argument("--no-parity-check", dest="parity_check", action="store_false", default=True,
                    help="skip the oracle replay of the timed frames (profiling runs)")
    ap.add_argument("--profile-step", type=int, default=-1,
                    help="bracket this timed step with cudaProfilerStart/Stop (for ncu --profile-from-start off; not a bench run)")
    ap.add_argument("--cpu-steps", type=int, default=6)
    ap.add_argument("--harness-frames", type=int, default=100, help="frames timed through the real ITMLib objects (0 = skip)")
    ap.add_argument("--hires-frames", type=int, default=24,
                    help="frames of the 4 mm roofline-stress stream (0 = skip; > 64 = the stream at length, e.g. 2000 for configs[4])")
    ap.add_argument("--decay-blocks", type=int, default=2000000, help="allocated blocks of the Decay() sweep, configs[3] (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (float32), to compare two builds on the same inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_own(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
