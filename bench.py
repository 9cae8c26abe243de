#!/usr/bin/env python
"""bench.py — frames/s of the active-window fusion hot path (BASELINE.json metric).

Workload "hall640" (BASELINE config[1]): synthetic 640x480 depth+label stream sweeping hall S2
(SURVEY.md §8d) into a 5 cm / 16^3-block map with MLE semantic fusion (L=20) and the tracking layer's
last_observed written (TSDF + semantic fusion only; K2/K3/M1 off). One lap of the trajectory is
rendered into HBM up front; a step = `--frames-per-step` consecutive frames (default: the whole lap) fused by
kb_integrate_frames (the C ABI the Khronos adaptor binds) in calls of `--batch` frames, device-resident images.

  value      whole-job frames/s, inputs already resident in HBM (CUDA events on the launch stream)
  e2e        same metric with HOST (pinned) images through the same C ABI, H2D inside the timed region
  roofline   dominant kernel (integrateKernel): algorithmic bytes per launch / mean launch duration
  cpu_baseline  the oracle port on this box's host cores over a bounded sample of the same stream

`--impl reference` times the CPU oracle port (the reference itself cannot be built here: it needs
Hydra/spatial_hash/Eigen/OpenCV, SURVEY.md §8c) on all host threads.
N > 1 (torchrun): the map shards by block hash, rank 0 broadcasts each step's frames over NCCL and
every rank integrates only the blocks it owns ("strong" scaling: total work is fixed).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

L_LABELS = 20
BYTES_PER_PIXEL_IN = 8  # depth f32 + label i32


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames-per-step", type=int, default=5000,
                    help="frames per step (default: one full lap, 12.3 GB of f32 input; 10 steps = ~0.4 s timed region)")
    ap.add_argument("--batch", type=int, default=0,
                    help="frames per kb_integrate_frames call; 0 (default) = the whole step in one call (the library fuses 32 frames "
                         "per kernel group inside a call and pipelines the groups); 1 = per-frame calls")
    ap.add_argument("--lap-frames", type=int, default=5000, help="frames in one lap of the trajectory (pool in HBM)")
    ap.add_argument("--max-blocks", type=int, default=90000)
    ap.add_argument("--cpu-sample-frames", type=int, default=5000,
                    help="upper bound on the frames of the cpu_baseline sample (it stops after --cpu-sample-seconds)")
    ap.add_argument("--cpu-sample-seconds", type=float, default=12.0, help="CPU work of the cpu_baseline sample")
    ap.add_argument("--ref-frames-per-step", type=int, default=256, help="--impl reference: frames per step")
    ap.add_argument("--e2e-frames", type=int, default=2048, help="frames of the e2e window (pinned host ring, ~0.1 s of PCIe traffic)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cull", action="store_true", help="disable the conservative depth culling (results identical)")
    ap.add_argument("--bcast", default="nccl", choices=["nccl", "multimem"],
                    help="N > 1 frame broadcast: 'nccl' = dist.broadcast; 'multimem' (experiment, unverified on hardware) = rank 0 stores "
                         "the step's frames once to the NVLS multicast mapping of a symmetric receive buffer (kb_multicast_copy)")
    ap.add_argument("--exchange", default="nccl", choices=["nccl", "peers"],
                    help="--workload dynamic, N > 1: 'nccl' = all-reduce / all-gathers; 'peers' (experiment, unverified on hardware) = "
                         "the producing kernels store into every rank's symmetric-memory buffers over NVLink, barriers only")
    ap.add_argument("--force-cull", action="store_true",
                    help="--workload dynamic: cull even single-frame calls (kb_set_culling(2)); results identical, 3 more launches per frame")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-legs", action="store_true", help="skip the secondary legs (output tick, per-frame pipeline on the hall stream, "
                    "next rows) of the N = 1 run")
    ap.add_argument("--wire", default="f32", choices=["f32", "compact", "f32u8"],
                    help="f32 = depth f32 + label i32 (hydra::InputData, 8 B/pixel; the headline); compact = u16 millimetre "
                         "depth + u8 labels (3 B/pixel, expanded on the device): what crosses PCIe / NVLink; f32u8 (N > 1 only, "
                         "experiment): lossless 5 B/pixel broadcast, depth f32 + labels narrowed to u8 on the ingest rank")
    ap.add_argument("--shard", default="cells", choices=["cells", "hash"],
                    help="N > 1: 'cells' = spatial cell sharding, stream striped over the ranks' pools, frames pulled over NVLink "
                         "only by the ranks whose cells they touch (khronos_b200/replay.py); 'hash' = round-1 design: per-block hash "
                         "sharding, every frame broadcast to every rank from rank 0")
    ap.add_argument("--cell-blocks", type=int, default=0,
                    help="--shard cells: cell side in blocks (16 = 12.8 m at 5 cm voxels); 0 (default) = pick among 12/16/20/24 the layout "
                         "with the fewest frames on the busiest rank for this trajectory (pose arithmetic only, kb_frame_owners)")
    ap.add_argument("--layout", default="auto", choices=["auto", "tiling", "bisect"],
                    help="--shard cells: 'tiling' = periodic tiling of square cells (--cell-blocks); 'bisect' = trajectory-aware table of "
                         "contiguous regions (replay.bisect_layout over kb_frame_cells, kb_set_shard_table); 'auto' (default) = whichever "
                         "puts the fewest frames on the busiest rank")
    ap.add_argument("--stripe", type=int, default=32, help="--shard cells: consecutive frames per rank in the striped pools")
    ap.add_argument("--gather", default="ce", choices=["ce", "sm", "bulk"],
                    help="--shard cells: transport of the NVLink pulls: copy engines, SM load/store kernel, cp.async.bulk kernel")
    ap.add_argument("--gather-ctas", type=int, default=32)
    ap.add_argument("--ingest", default="routed", choices=["routed", "striped", "rank0"],
                    help="--shard cells: where the stream is resident. routed (default): the host, which knows the poses, hands every "
                         "32-frame chunk to a rank whose cells it touches (one delivery per frame is local); striped: chunks dealt round "
                         "robin; rank0: everything on rank 0 (its NVLink egress then bounds the exchange)")
    ap.add_argument("--fuse-ctas-per-sm", type=int, default=0,
                    help="N > 1: resident fusion CTAs per SM (KB_FUSE_CTAS_PER_SM; 0 = library default = full occupancy). Fewer CTAs leave "
                         "registers for the next batch's block selection / culling kernels to run beside the fusion kernel")
    ap.add_argument("--small", action="store_true", help="tiny configuration for functional checks")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="1 GPU, hall workloads: after the timed steps, write the map they produced as DIR/<name>.npy (every "
                         "block index, and the voxels of a fixed seeded sample of the blocks), so that two builds can be compared")
    ap.add_argument("--workload", default="hall640", choices=["hall640", "hall1280", "dynamic"],
                    help="hall640 = BASELINE config[1] (fusion only, the headline, used for every --gpus N); hall1280 = "
                         "config[3] shapes (1280x720, 2 cm voxels: ~20x the voxel work per frame) for the sharded "
                         "scaling study; dynamic = config[2]: per-frame pipeline with motion detection + tracking")
    return ap.parse_args()


def workload(args):
    from khronos_b200 import synthetic as syn
    if args.small:
        cam = syn.make_camera(160, 120, 80.0, 80.0)
        scene = syn.hall_scene(L_LABELS, size=(20.0, 16.0, 6.0))
        poses, stamps = syn.sweep_trajectory(args.lap_frames, size=(20.0, 16.0), margin=4.0, lanes=3, yaw_turns=6.0)
    elif args.workload == "hall1280":
        cam = syn.make_camera(1280, 720, 640.0, 640.0)
        scene = syn.hall_scene(L_LABELS, size=(30.0, 20.0, 6.0))
        poses, stamps = syn.sweep_trajectory(args.lap_frames, size=(30.0, 20.0), margin=5.0, lanes=3, yaw_turns=10.0)
    else:
        cam = syn.make_camera()
        scene = syn.hall_scene(L_LABELS)
        poses, stamps = syn.sweep_trajectory(args.lap_frames)
    return cam, scene, poses, stamps


def algorithmic_bytes(nv, nsem, nblk, pixels, lp=20, bpp=BYTES_PER_PIXEL_IN):
    """Byte model (DESIGN.md §4): per integrated voxel 8 B read + 8 B write of {distance, weight} and a
    4 B last_observed write; per semantic update Lp*4 B read + write of the likelihood row and a 2 B
    label read + write; the frame's depth + label images once; 16 B of hash/index per visited block."""
    return nv * (8 + 8 + 4) + nsem * (2 * 4 * lp + 4) + pixels * bpp + nblk * 16


class ClockSampler:
    """Samples nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md). The timed region of the
    default run is ~0.1 s, so nvidia-smi is started early (before the last warm-up step: its start-up latency is of
    that order) with a 20 ms period, every sample is stamped on arrival, and stop(t0, t1) keeps the samples that fell
    inside the timed window [t0, t1] (perf_counter seconds)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0, period_ms=20):
        self.index, self.rows, self.proc, self.period_ms = index, [], None, period_ms

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", str(self.period_ms)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def stop(self, t0=None, t1=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        rows = [(t, r) for t, r in list(self.rows) if len(r) >= 6]
        late = False
        if not rows:  # the sampler never produced a line (slow start): one synchronous query right after the region
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=20).stdout
                rows = [(time.perf_counter(), [x.strip() for x in ln.split(",")]) for ln in out.splitlines() if ln.count(",") >= 5]
                late = bool(rows)
            except Exception:
                rows = []
        inside = [r for t, r in rows if (t0 is None or t >= t0) and (t1 is None or t <= t1 + 0.5 * self.period_ms * 1e-3)]
        note = None
        if not inside and rows and t0 is not None:  # region shorter than the sampling period: nearest samples around it
            mid = 0.5 * (t0 + t1)
            inside = [r for _, r in sorted(rows, key=lambda tr: abs(tr[0] - mid))[:2]]
            note = "no sample landed inside the timed window; the 2 nearest samples are reported"
        num = lambda x: x.replace(".", "").isdigit()
        sm = [float(r[0]) for r in inside if num(r[0])]
        mx = [float(r[1]) for r in inside if num(r[1])]
        reasons = set()
        for r in inside:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        out = {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
               "reasons": sorted(reasons), "samples": len(sm), "samples_total": len(rows)}
        if late:
            note = "sampler produced no line in time; one query taken right after the timed region"
        if note:
            out["note"] = note
        return out


def map_configs(args):
    from khronos_b200 import capi
    vs, tr = (0.02, 0.06) if args.workload == "hall1280" else (0.05, 0.15)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    mb = args.max_blocks if not args.small else 8192
    msem = 0
    if args.workload == "hall1280" and not args.small:
        mb = max(args.max_blocks, 420000) // world + 20000   # block-hash shard: 1/N of the map per GPU
        msem = mb // 2
    mc = capi.default_map_config(voxel_size=vs, vps=16, trunc=tr, with_semantics=True, with_tracking=True,
                                 max_blocks=mb, max_semantic_blocks=msem)
    ic = capi.default_integrator_config(semantic_mode=capi.SEM_MLE, num_labels=L_LABELS)
    return mc, ic


def run_cpu(args, cam, frames_host, poses, stamps, n_frames, threads=-1):
    """Times the oracle port on host cores over frames [0, n_frames). Returns (fps, cores, seconds)."""
    fps, cores, dt, _ = run_cpu_stream(args, cam, lambda i, k: (frames_host[0][i:i + k], frames_host[1][i:i + k]),
                                       poses, stamps, n_frames, float("inf"), threads)
    return fps, cores, dt


def run_cpu_stream(args, cam, chunk_fn, poses, stamps, max_frames, budget_s, threads=-1, chunk=128):
    """Oracle port over consecutive frames from the start of the stream into an empty map, fetched in chunks
    (chunk_fn(i, k) -> host depth/label arrays of frames [i, i+k)) until `budget_s` seconds of integration time
    or `max_frames` frames. Only the integrate calls are timed. Returns (fps, cores, seconds, frames)."""
    from khronos_b200 import capi
    lib = ctypes.CDLL(os.path.join(ROOT, "oracle", "liboracle.so"))
    mc, ic = map_configs(args)
    ic.num_threads = threads
    h = capi.MapHandle(lib, "ko_", mc, ic, capi.default_tracking_config(), None)
    h.set_camera(cam)
    n, dt = 0, 0.0
    while n < max_frames and dt < budget_s:
        k = min(chunk, max_frames - n)
        d, l = chunk_fn(n, k)
        fr = [h.make_frame(d[j], poses[n + j], stamps[n + j], label=l[j]) for j in range(k)]
        t0 = time.perf_counter()
        for f in fr:
            h.integrate_frame(f, want_stats=False)
        dt += time.perf_counter() - t0
        n += k
    cores = os.cpu_count() if threads <= 0 else threads
    h.close()
    return n / dt, cores, dt, n


def best_cpu_threads(args, cam, frames_host, poses, sel, n_probe=12):
    """The oracle spawns its workers per frame like the reference; on many-core hosts fewer threads than
    hardware_concurrency can be faster. Be generous to the CPU arm: probe and keep the best."""
    best, best_fps = None, 0.0
    ncpu = os.cpu_count() or 1
    for t in sorted({min(ncpu, x) for x in (8, 16, 32, 64, 128, ncpu)}):
        st = [1_000_000_000 + k * 33_333_333 for k in range(n_probe)]
        fps, _, _ = run_cpu(args, cam, (frames_host[0][:n_probe], frames_host[1][:n_probe]),
                            [poses[i] for i in sel[:n_probe]], st, n_probe, threads=t)
        if fps > best_fps:
            best, best_fps = t, fps
    return best


def main_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port; the real binary is unbuildable
    here) on all host threads, each step a bounded sample of the same stream."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from khronos_b200 import synthetic as syn
    cam, scene, poses, stamps = workload(args)
    per_step = max(4, args.ref_frames_per_step if not args.small else 8)
    n = per_step * (args.steps + args.warmup)
    stride = 1  # a contiguous chunk of the same stream (same inter-frame overlap as the GPU arm sees)
    sel = [i % len(poses) for i in range(n)]
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    d, l = syn.render_stream(scene, cam, [poses[i] for i in sel], [stamps[i] for i in sel], device=dev, dtype=torch.float32)
    d, l = d.cpu().numpy(), l.cpu().numpy()
    from khronos_b200 import capi
    lib = ctypes.CDLL(os.path.join(ROOT, "oracle", "liboracle.so"))
    mc, ic = map_configs(args)
    ic.num_threads = best_cpu_threads(args, cam, (d, l), poses, sel)
    h = capi.MapHandle(lib, "ko_", mc, ic, capi.default_tracking_config(), None)
    h.set_camera(cam)
    # stamps must increase along the sampled sequence
    fr = [h.make_frame(d[k], poses[i], 1_000_000_000 + k * 33_333_333, label=l[k]) for k, i in enumerate(sel)]
    for f in fr[: per_step * args.warmup]:
        h.integrate_frame(f, want_stats=False)
    t0 = time.perf_counter()
    for f in fr[per_step * args.warmup:]:
        h.integrate_frame(f, want_stats=False)
    dt = time.perf_counter() - t0
    fps = per_step * args.steps / dt
    out = {
        "impl": "reference", "metric": "rgbd_frames_per_sec_integrated", "value": fps, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "hall640" if not args.small else "hall160-small", "image": [cam.width, cam.height],
                   "voxel_size": 0.05, "voxels_per_side": 16, "semantics": "MLE L=20",
                   "frames_per_step": per_step},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": ic.num_threads, "kind": "port",
                         "sample": f"{per_step} consecutive frames/step from the start of the lap, oracle port, best "
                                   f"thread count of a sweep up to {os.cpu_count()} host threads "
                                   f"(reference needs Hydra/Eigen/OpenCV: unbuildable here)"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(out)


def main_dynamic(args):
    """BASELINE config[2]: per-frame pipeline of ActiveWindow::spinOnce (active_window.cpp:118-174) on one
    GPU: kb_detect_motion -> kb_integrate_frame(mask = dynamic image) -> kb_update_tracking, room scene S1,
    slow orbit, a box that stays ~2.2 m in front of the camera covers ~20 % of the pixels after a 2 s burn-in.
    Frames are resident in HBM; the dynamic image makes a host round trip (M2-M4 cluster on the host)."""
    import torch
    import khronos_b200 as kb
    from khronos_b200 import capi, synthetic as syn
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    F, K, Wm = min(args.frames_per_step, 150), args.steps, args.warmup
    n = F * (K + Wm)
    cam = syn.make_camera() if not args.small else syn.make_camera(160, 120, 80.0, 80.0)
    scene = syn.room_scene(L_LABELS)
    poses, stamps = syn.orbit_trajectory(n, laps=n / 3000.0)
    extra = syn.companion_cuboids(poses)
    depth, label = syn.render_stream(scene, cam, poses, stamps, device=dev, dtype=torch.float32, extra=extra)
    mc, ic = map_configs(args)
    mot = capi.default_motion_config(min_cluster_size=500 if not args.small else 30, min_separation_distance=2.0)
    h = kb.create_map(mc, ic, capi.default_tracking_config(), mot, device=0)
    h.set_camera(cam)
    if args.force_cull:
        h.set_culling(2)
    flagged = []
    img_host = torch.zeros((cam.height, cam.width), dtype=torch.int32, pin_memory=True)  # FrameData::dynamic_image
    img_ptr = ctypes.c_void_p(img_host.data_ptr())
    spin = h._fn("spin_once")
    hptr = h._h

    frames = [h.make_frame(depth[i].data_ptr(), poses[i], stamps[i], label=label[i].data_ptr(), memory=capi.MEM_DEVICE)
              for i in range(n)]

    def run_frame(i):
        f = frames[i]
        ns, nc = ctypes.c_int32(0), ctypes.c_int32(0)
        # detect -> integrate(mask = dynamic image) -> track, one host round trip (dynamic image -> pinned host)
        st = spin(hptr, ctypes.byref(f), img_ptr, ctypes.byref(ns), ctypes.byref(nc))
        if st != 0:
            raise RuntimeError(f"kb_spin_once failed: {st}")
        return nc.value

    for i in range(Wm * F):
        run_frame(i)
    h.synchronize()
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    t0 = time.perf_counter()
    for i in range(Wm * F, n):
        flagged.append(run_frame(i))  # number of clusters; no host-side image processing inside the timed region
    h.synchronize()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    clocks = sampler.stop(t0, t0 + dt)
    tot = h.get_totals()
    # CPU arm of the same pipeline on a bounded sample: the oracle port replays the first frames (burn-in + the first
    # dynamic frames) and is timed on the frames in which it finds clusters
    cpu = None
    if not args.no_cpu_baseline:
        n_c = min(n, 60 + 40)
        lib = ctypes.CDLL(os.path.join(ROOT, "oracle", "liboracle.so"))
        # 32 worker threads: the best of the fusion arm's thread sweeps on this pool's hosts (the oracle spawns its workers per
        # frame like the reference; hardware_concurrency = 128 is slower)
        nthr = min(32, os.cpu_count() or 1)
        ic_c, _ = map_configs(args)[1], None
        ic_c.num_threads = nthr
        mot_c = capi.default_motion_config(min_cluster_size=mot.min_cluster_size, min_separation_distance=2.0, num_threads=nthr)
        oh = capi.MapHandle(lib, "ko_", mc, ic_c, capi.default_tracking_config(num_threads=nthr), mot_c)
        oh.set_camera(cam)
        dh, lh = depth[:n_c].cpu().numpy(), label[:n_c].cpu().numpy()
        times = []
        for i in range(n_c):
            fo = oh.make_frame(dh[i], poses[i], stamps[i], label=lh[i])
            t1 = time.perf_counter()
            _, _, nc_i = oh.spin_once(fo)
            if nc_i:
                times.append(time.perf_counter() - t1)
        if times:
            cpu = {"value": len(times) / sum(times), "unit": "frames/s", "cores": nthr, "kind": "port",
                   "sample": f"{len(times)} dynamic frames after a 60-frame burn-in, oracle port (detect + integrate + track)"}
    out = {
        "metric": "rgbd_frames_per_sec_integrated", "value": K * F / dt, "unit": "frames/s", "n_gpus": 1, "steps": K,
        "warmup": Wm, "ms_per_step": dt / K * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "room640-dynamic (BASELINE config[2])", "image": [cam.width, cam.height],
                   "voxel_size": 0.05, "voxels_per_side": 16, "semantics": f"MLE L={L_LABELS}", "frames_per_step": F,
                   "pipeline": "kb_spin_once per frame (= kb_detect_motion + kb_integrate_frame(mask) + kb_update_tracking, one host round trip)",
                   "live_blocks": tot.total_blocks},
        "per_frame": {"frames_with_clusters": int(sum(1 for x in flagged if x > 0)),
                      "flagged_pixel_fraction_last_frame": float((img_host.numpy() > 0).mean())},
        "roofline": None, "cpu_baseline": cpu, "e2e": None, "gpu_launches": 16 * K * F, "clocks": clocks,
    }
    emit(out)


def main_dynamic_sharded(args):
    """BASELINE config[2] on N GPUs (torchrun): the same per-frame pipeline as main_dynamic over a block-hash sharded map.
    Per frame rank 0 broadcasts depth + label (NCCL), then every rank runs khronos_b200.distributed.ShardedActiveWindow.
    spin_once: M1 local lookup -> all-reduce(MAX) of the pixel flags -> replicated M2-M4 -> sharded K0/K1 with the dynamic
    mask -> K2 -> two all-gathers (pending blocks, free masks) -> K3; one host round trip per frame (counts)."""
    import torch
    import torch.distributed as dist
    import khronos_b200 as kb
    from khronos_b200 import capi, synthetic as syn, distributed as kd
    world, rank = int(os.environ["WORLD_SIZE"]), int(os.environ["RANK"])
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist.init_process_group("nccl", device_id=dev)
    F, K, Wm = min(args.frames_per_step, 150), args.steps, args.warmup
    n = F * (K + Wm)
    cam = syn.make_camera() if not args.small else syn.make_camera(160, 120, 80.0, 80.0)
    scene = syn.room_scene(L_LABELS)
    poses, stamps = syn.orbit_trajectory(n, laps=n / 3000.0)
    H, W = cam.height, cam.width
    if rank == 0:
        extra = syn.companion_cuboids(poses)
        depth, label = syn.render_stream(scene, cam, poses, stamps, device=dev, dtype=torch.float32, extra=extra)
    rx = torch.zeros((2, H, W), dtype=torch.int32, device=dev)  # packed (depth bits, label): one broadcast per frame
    rx_depth, rx_label = rx[0].view(torch.float32), rx[1]
    mc, ic = map_configs(args)
    mot = capi.default_motion_config(min_cluster_size=500 if not args.small else 30, min_separation_distance=2.0)
    h = kb.create_map(mc, ic, capi.default_tracking_config(), mot, device=local_rank)
    h.set_camera(cam)
    h.set_shard(rank, world)
    # exchange buffers are shipped whole (no host round trip to learn the fill): size them for this workload. Counted on the
    # emulated build at 640x480: ~172 pending blocks per frame over all ranks; published halo blocks per rank 147 (N = 2) / 42 (N = 8)
    h.set_shard_capacity(256, 512)
    if args.exchange == "peers":
        win = kd.PeerShardedActiveWindow([h], kd.SymmMemPeers(device=dev), device=dev)
    else:
        win = kd.ShardedActiveWindow([h], kd.DistComm(world), device=dev)
    frames = [h.make_frame(rx_depth.data_ptr(), poses[i], stamps[i], label=rx_label.data_ptr(), memory=capi.MEM_DEVICE)
              for i in range(n)]
    clusters = []

    def run_frame(i):
        if rank == 0:
            rx_depth.copy_(depth[i])
            rx_label.copy_(label[i])
        dist.broadcast(rx, 0)
        (_, ns, nc), = win.spin_once([frames[i]], want_image=False)
        return nc

    for i in range(Wm * F):
        run_frame(i)
    dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    t0 = time.perf_counter()
    for i in range(Wm * F, n):
        clusters.append(run_frame(i))
    torch.cuda.synchronize()
    dist.barrier()
    dt = time.perf_counter() - t0
    clocks = sampler.stop(t0, t0 + dt) if rank == 0 else None
    t = torch.tensor([dt], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt = float(t.item())
    tot = h.get_totals()
    if tot.capacity_exceeded:
        raise SystemExit("bench.py: a shard exchange buffer / block pool overflowed (capacity_exceeded): results incomplete")
    blocks = torch.tensor([float(tot.total_blocks)], device=dev, dtype=torch.float64)
    dist.all_reduce(blocks)
    if rank == 0:
        pb, hb, fb = h.shard_buffer_sizes()
        out = {
            "metric": "rgbd_frames_per_sec_integrated", "value": K * F / dt, "unit": "frames/s", "n_gpus": world, "steps": K,
            "warmup": Wm, "ms_per_step": dt / K * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "room640-dynamic (BASELINE config[2])", "image": [W, H], "voxel_size": 0.05,
                       "voxels_per_side": 16, "semantics": f"MLE L={L_LABELS}", "frames_per_step": F,
                       "pipeline": ("per frame: NCCL frame broadcast + ShardedActiveWindow.spin_once (pixel-flag all-reduce, 2 halo "
                                    "all-gathers, one host round trip)" if args.exchange == "nccl" else
                                    "per frame: NCCL frame broadcast + PeerShardedActiveWindow.spin_once (producers store into "
                                    "every rank's symmetric-memory buffers, 3 barriers, one host round trip)"),
                       "parallelism": "block-hash shard x%d" % world, "live_blocks_all_ranks": int(blocks.item()),
                       "exchange_bytes_per_frame_per_rank": {"pixel_flags": fb, "pending": pb, "halo": hb}},
            "per_frame": {"frames_with_clusters": int(sum(1 for x in clusters if x > 0))},
            "roofline": None, "cpu_baseline": None, "e2e": None, "gpu_launches": 24 * K * F, "clocks": clocks,
        }
        emit(out)
    dist.destroy_process_group()


_REAL_STDOUT = None


def quiet_stdout():
    """Libraries (NCCL, torch) print banners on fd 1; the contract is ONE JSON line on stdout. Everything is routed
    to stderr until emit() restores the real stdout for the result line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(obj), flush=True)


def load_capture():
    """Per-launch DRAM traffic / issue utilisation of the dominant kernel from THIS round's `ncu --set full` capture
    (profiles/r2_fuse_capture.json, written by tools/ncu_digest.py from the committed csv export). None if absent."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r2_fuse_capture.json")))
    except Exception:
        return None


def hbm_peak():
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(peaks["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        return 6650.0, "fallback 6650 (of fallback)"


GROUP = 32  # frames fused per kernel group inside a kb_integrate_frames call (csrc/kb_kernels.cuh kMaxBatch)


def n_groups(n):
    return (n + GROUP - 1) // GROUP


def roofline_block(args, B, n_calls, gpu_ms, sampled_us, nv, nsem, nblk, n_frames, P, bpp, world=1):
    """roofline of the dominant kernel group (one kb_integrate_frames call = tile pyramid + K0 + K0b + item lists + fuse
    kernel for B frames). achieved = algorithmic bytes of the timed region / device time of the timed region (every
    launch inside it belongs to such a group, and with the pipelined prologue the groups overlap, so the region average
    is the only well-defined per-group duration); launch_us_sampled = CUDA events around individual calls."""
    peak, src = hbm_peak()
    total_bytes = algorithmic_bytes(nv, nsem, nblk, n_frames * P, bpp=bpp)
    per_launch = total_bytes / max(n_calls, 1)
    avg_us = gpu_ms * 1e3 / max(n_calls, 1)
    achieved = total_bytes / (gpu_ms * 1e-3) / 1e9
    cap = load_capture()
    traffic = issue = None
    if cap and cap.get("frames_per_launch") == B and args.workload == "hall640" and not args.small and world == 1:
        traffic = cap.get("dram_bytes_per_launch_group")
        issue = cap.get("fuse_issue_slot_utilization_pct")
    out = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
           "kernel": "fuseKernel<16> + its prologue (tileMax, tilePyramid, selectBlocks, itemCull, itemCompact): one group per %d frames" % B,
           "launch_us": avg_us, "launch_us_sampled": sampled_us, "algorithmic_bytes_per_launch": per_launch,
           "peak_source": src,
           "note": "the kernel is issue-bound, not HBM-bound (DRAM traffic is below the algorithmic bytes: the working set is L2 "
                   "resident); frac_dram = measured DRAM bytes / time / peak, issue_slot_utilization from the same ncu capture"}
    if traffic:
        out["frac_dram"] = traffic / (avg_us * 1e-6) / 1e9 / peak
    if issue is not None:
        out["issue_slot_utilization_pct"] = issue
    return out


def combine_checksums(parts):
    """parts: per-rank (sum, xor, blocks, observed) -> the unsharded map's checksum (sums wrap mod 2^64)."""
    m = (1 << 64) - 1
    x = 0
    for p in parts:
        x ^= int(p[1])
    return {"sum": "%016x" % (sum(int(p[0]) for p in parts) & m), "xor": "%016x" % x,
            "blocks": int(sum(int(p[2]) for p in parts)), "observed_voxels": int(sum(int(p[3]) for p in parts))}


DUMP_SAMPLE_BLOCKS = 512  # voxels of 512 blocks: 40 MB, inside the 64 MB the dump may take
DUMP_SEED = 0


def dump_outputs(h, out_dir):
    """Writes the map as a caller reads it back (kb_export_blocks, blocks ascending in (x, y, z)): the index of every block,
    and the TSDF, semantic label (-1 where the voxel has none) and last_observed stamp of every voxel of a fixed seeded
    sample of the blocks. The sample is drawn by position in the sorted block list, so two builds that compute the same
    map dump the same blocks. One field is exported per call to bound host memory (the whole map is GBs)."""
    from khronos_b200 import capi
    n, V = h.num_blocks(), h.V

    def field(name, dtype, width):
        a = np.zeros((n, width), dtype)
        ex = capi.BlockExport()
        setattr(ex, name, a.ctypes.data)
        nw = ctypes.c_int32(0)
        if n:
            h._check(h._fn("export_blocks")(h._h, capi.EXPORT_ALL, n, ctypes.byref(ex), ctypes.byref(nw)))
            assert nw.value == n
        return a

    index = field("block_index", np.int32, 3)
    sel = np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=min(DUMP_SAMPLE_BLOCKS, n), replace=False))
    empty = field("semantic_empty", np.uint8, V)[sel]
    out = {
        "block_index": index.astype(np.float64),
        "sample_block_index": index[sel].astype(np.float64),
        "sample_distance": field("distance", np.float32, V)[sel],
        "sample_weight": field("weight", np.float32, V)[sel],
        "sample_semantic_label": np.where(empty != 0, -1.0, field("semantic_label", np.uint32, V)[sel]).astype(np.float32),
        "sample_last_observed_ns": field("last_observed", np.uint64, V)[sel].astype(np.float64),  # exact below 2^53 ns
    }
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main_hall_cells(args, world, rank, local_rank, dev):
    """N > 1, --shard cells (khronos_b200/replay.py): cell-sharded map, stream striped over the ranks' frame pools, every
    rank pulls the frames whose frustum touches its cells over NVLink (CUDA IPC peer mappings) and fuses its sub-sequence
    in stream order, double buffered against the pulls of the next step. Returns None after printing the result line,
    or a string (reason) when peer memory cannot be set up, in which case the caller falls back to --shard hash."""
    import torch
    import torch.distributed as dist
    import khronos_b200 as kb
    from khronos_b200 import capi, synthetic as syn
    from khronos_b200.replay import PeerPools, StripedSchedule, rank_grid

    lib = kb.lib()
    F, K, Wm = args.frames_per_step, args.steps, args.warmup
    if args.small:
        F = min(F, 64)
        args.lap_frames = min(args.lap_frames, 256)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    cam, scene, poses, stamps = workload(args)
    lap, H, W = len(poses), cam.height, cam.width
    P = H * W
    bpp = BYTES_PER_PIXEL_IN
    if args.fuse_ctas_per_sm > 0:
        os.environ["KB_FUSE_CTAS_PER_SM"] = str(args.fuse_ctas_per_sm)  # read by kb_create
    mc, ic = map_configs(args)
    h = kb.create_map(mc, ic, capi.default_tracking_config(), None, device=local_rank)
    h.set_camera(cam)
    if args.no_cull:
        h.set_culling(False)
    gx, gy = rank_grid(world)
    # which ranks need which frame: pure pose arithmetic (kb_frame_owners), identical on every rank. The per-batch cost of a
    # rank is dominated by fixed work per frame it receives (tile pyramid, block selection, the critical path of the fusion
    # kernel), so the layout with the fewest frames on the busiest rank wins (measured: profiles/r2_multigpu_summary.txt).
    probe_frames = [h.make_frame(None, poses[g], stamps[g]) for g in range(lap)]
    frames_of = lambda m_: [int(((m_ >> r) & 1).sum()) for r in range(world)]
    layouts = {}
    if args.layout in ("auto", "tiling"):
        for cb in ([args.cell_blocks] if args.cell_blocks > 0 else [12, 16, 20, 24]):
            h.set_shard_cells(rank, world, cb, gx, gy)
            m_ = h.frame_owners(probe_frames)
            layouts[("tiling", cb)] = (max(frames_of(m_)), m_, None)
    if args.layout in ("auto", "bisect"):
        from khronos_b200.replay import bisect_layout
        tcell = 4  # table granularity: 4 x 4 blocks (3.2 m at 5 cm voxels); regions are contiguous rectangles of such cells
        bsz = mc.voxel_size * 16 * tcell
        reach = cam.max_range + 2 * mc.voxel_size * 16
        px = np.array([np.asarray(T, np.float64).reshape(4, 4)[0, 3] for T in poses])
        py = np.array([np.asarray(T, np.float64).reshape(4, 4)[1, 3] for T in poses])
        tox, toy = int(np.floor((px.min() - reach) / bsz)), int(np.floor((py.min() - reach) / bsz))
        tw, th = int(np.floor((px.max() + reach) / bsz)) - tox + 1, int(np.floor((py.max() + reach) / bsz)) - toy + 1
        touched = h.frame_cells(probe_frames, tcell, (tox, toy), tw, th)
        table = bisect_layout(touched, world)
        h.set_shard_table(rank, world, tcell, (tox, toy), table)
        m_ = h.frame_owners(probe_frames)
        layouts[("bisect", tcell)] = (max(frames_of(m_)), m_, ((tox, toy), table))
    choice = min(layouts, key=lambda k: (layouts[k][0], k[0] != "bisect", -k[1]))
    masks = layouts[choice][1]
    if choice[0] == "bisect":
        h.set_shard_table(rank, world, choice[1], layouts[choice][2][0], layouts[choice][2][1])
        layout_desc = ("trajectory-aware table of %d contiguous regions (recursive bisection of %d x %d cells of %d x %d blocks = %.1f m by "
                       "frames-per-region, kb_set_shard_table)" % (world, layouts[choice][2][1].shape[1], layouts[choice][2][1].shape[0],
                                                                    choice[1], choice[1], choice[1] * mc.voxel_size * 16))
    else:
        h.set_shard_cells(rank, world, choice[1], gx, gy)
        layout_desc = "cells of %d x %d blocks = %.1f m, %d x %d rank tiling" % (choice[1], choice[1], choice[1] * mc.voxel_size * 16, gx, gy)
    args.cell_blocks = choice[1]
    layout_proxy = {"%s-%d" % k: v[0] for k, v in layouts.items()}
    stripe = args.stripe
    if args.ingest == "rank0":
        homes = np.zeros(lap, np.int32)
    elif args.ingest == "routed":
        from khronos_b200.replay import route_homes
        homes = route_homes(masks, world, stripe)
    else:
        homes = None
    sched = StripedSchedule(world, rank, stripe, homes=homes)
    res = sched.resident(lap)

    # ---- this rank's part of the stream, rendered straight into its (IPC-shareable) pool
    t_render = time.perf_counter()
    note = None
    try:
        pool = PeerPools(lib, local_rank, len(res), H, W)
        dv, lv = pool.views(torch, dev)
        t0s = stamps[0]
        for li, g in enumerate(res):
            d, l = syn.render(scene, cam, poses[g], (stamps[g] - t0s) * 1e-9, device=dev, dtype=torch.float32)
            dv[li].copy_(d)
            lv[li].copy_(l)
        torch.cuda.synchronize()
        hb = torch.tensor(list(pool.export_handle()), dtype=torch.uint8, device=dev)
        hs_all = [torch.empty_like(hb) for _ in range(world)]
        dist.all_gather(hs_all, hb)
        nres = torch.tensor([len(res)], dtype=torch.int64, device=dev)
        n_all = [torch.empty_like(nres) for _ in range(world)]
        dist.all_gather(n_all, nres)
        for q in range(world):
            if q != rank:
                pool.open_peer(q, bytes(hs_all[q].cpu().tolist()), int(n_all[q].item()))
    except Exception as e:  # noqa: BLE001 - any failure of the peer set-up selects the fallback on ALL ranks
        note = "peer memory unavailable (%s)" % str(e)[:160]
    flag = torch.tensor([1 if note else 0], device=dev)
    dist.all_reduce(flag)
    if int(flag.item()):
        h.close()
        return note or "peer memory unavailable on another rank"
    t_render = time.perf_counter() - t_render

    stream = torch.cuda.Stream(device=dev)
    xstream = torch.cuda.Stream(device=dev)
    h.set_stream(stream.cuda_stream)
    B = F if args.batch <= 0 else max(1, min(args.batch, F))  # frames per kb_integrate_frames call

    def frame_index(step, j):
        return (step * F + j) % lap

    def stamp_of(step, j):
        return 1_000_000_000 + (step * F + j) * 33_333_333

    # ---- schedule: pulls and frame descriptors — all outside the timed region
    plans = {s: sched.plan([frame_index(s, j) for j in range(F)], masks) for s in range(Wm + K)}
    cap = max(1, max(p.n_remote for p in plans.values()))
    rx = [PeerPools(lib, local_rank, cap, H, W) for _ in range(2)]
    mode = {"ce": 0, "sm": 1, "bulk": 2}[args.gather]
    gplans = {s: pool.gather_plan(plans[s].ranges, rx[s % 2].ptr, cap) for s in plans}
    calls = {}
    for s, pl in plans.items():
        fr = []
        for j, g, slot in pl.mine:
            base, cnt, i = (rx[s % 2].ptr, cap, slot) if slot >= 0 else (pool.ptr, pool.n, -slot - 1)
            fr.append(h.make_frame(pool.depth_ptr(base, cnt, i), poses[g], stamp_of(s, j), label=pool.label_ptr(base, cnt, i),
                                   memory=capi.MEM_DEVICE))
        calls[s] = [((capi.Frame * len(fr[k:k + B]))(*fr[k:k + B]), len(fr[k:k + B])) for k in range(0, len(fr), B)]
    integrate_n = h._fn("integrate_frames")
    hptr = h._h
    ready, gather_ev, buf_free, issued = {}, {}, [None, None], set()

    def issue_gather(s):
        b = s % 2
        if buf_free[b] is not None:
            xstream.wait_event(buf_free[b])  # the fusion of step s-2 no longer reads rx[b]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(xstream)
        pool.run(gplans[s], mode, args.gather_ctas, xstream.cuda_stream)
        e1.record(xstream)
        gather_ev[s] = (e0, e1)
        ready[s] = e1
        issued.add(s)

    def run_step(s, last_of_phase, samples=None):
        if s not in issued:
            issue_gather(s)
        if not last_of_phase and (s + 1) in plans and (s + 1) not in issued:
            issue_gather(s + 1)  # overlaps this step's fusion
        stream.wait_event(ready[s])
        with torch.cuda.stream(stream):
            for k, (arr, n) in enumerate(calls[s]):
                if samples is not None and n >= GROUP:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    st = integrate_n(hptr, arr, n, 1, None)
                    e1.record(stream)
                    samples.append((e0, e1, n))
                else:
                    st = integrate_n(hptr, arr, n, 1, None)
                if st != 0:
                    raise RuntimeError(f"kb_integrate_frames failed: {st}")
        ev = torch.cuda.Event()
        ev.record(stream)
        buf_free[s % 2] = ev

    def barrier():
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()

    for s in range(Wm):
        run_step(s, s == Wm - 1)
    barrier()
    t64_0 = h.get_totals64()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    samples = []
    wall0 = time.perf_counter()
    ev0.record(stream)
    for s in range(Wm, Wm + K):
        run_step(s, s == Wm + K - 1, samples)
    ev1.record(stream)
    torch.cuda.synchronize()
    busy_ms = ev0.elapsed_time(ev1)
    dist.barrier()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop(wall0, wall0 + wall) if rank == 0 else None
    t = torch.tensor([busy_ms], device=dev, dtype=torch.float64)
    all_busy = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(all_busy, t)
    busy = [float(x.item()) for x in all_busy]
    gpu_ms = max(busy)  # device time of the timed region, max over ranks
    t64_1 = h.get_totals64()
    if t64_1.capacity_exceeded:
        raise SystemExit("bench.py: block pool exhausted (capacity_exceeded): results incomplete")
    cs = h.map_checksum()
    n_frames = K * F
    my_frames = sum(len(plans[s].mine) for s in range(Wm, Wm + K))
    my_remote = sum(plans[s].n_remote for s in range(Wm, Wm + K))
    g_ms = sum(gather_ev[s][0].elapsed_time(gather_ev[s][1]) for s in range(Wm, Wm + K))
    g_bytes = sum(pool.plan_bytes(gplans[s]) for s in range(Wm, Wm + K))
    nv = t64_1.voxels_updated - t64_0.voxels_updated
    nsem = t64_1.voxels_semantic - t64_0.voxels_semantic
    nblk = t64_1.blocks_in_frustum - t64_0.blocks_in_frustum
    stats = torch.tensor([float(nv), float(nsem), float(nblk), float(my_frames), float(my_remote), g_ms, float(g_bytes),
                          float(t64_1.total_blocks)], device=dev, dtype=torch.float64)
    all_stats = [torch.empty_like(stats) for _ in range(world)]
    dist.all_gather(all_stats, stats)
    cst = torch.tensor([int(c) - (1 << 64) if int(c) >= (1 << 63) else int(c) for c in cs], device=dev, dtype=torch.int64)
    all_cs = [torch.empty_like(cst) for _ in range(world)]
    dist.all_gather(all_cs, cst)

    # ---- e2e at N GPUs: every rank integrates the frames it needs from its OWN pinned host memory over its own PCIe link
    # (the production ingest: the host knows the poses, so it hands each frame only to the ranks whose cells it touches)
    e2e = None
    if not args.no_e2e:
        n_e = min(args.e2e_frames, lap) if not args.small else min(64, lap)
        step_e = Wm + K + 2
        need = [(j, frame_index(step_e, j)) for j in range(n_e) if (int(masks[frame_index(step_e, j)]) >> rank) & 1]
        hd = torch.empty((max(len(need), 1), H, W), dtype=torch.float32, pin_memory=True)
        hl = torch.empty((max(len(need), 1), H, W), dtype=torch.int32, pin_memory=True)
        for k, (j, g) in enumerate(need):
            d, l = syn.render(scene, cam, poses[g], 0.0, device=dev, dtype=torch.float32)
            hd[k].copy_(d)
            hl[k].copy_(l)
        torch.cuda.synchronize()
        fr = [h.make_frame(hd[k].data_ptr(), poses[g], stamp_of(step_e, j), label=hl[k].data_ptr(), memory=capi.MEM_HOST_ASYNC)
              for k, (j, g) in enumerate(need)]
        ecalls = [((capi.Frame * len(fr[k:k + B]))(*fr[k:k + B]), len(fr[k:k + B])) for k in range(0, len(fr), B)]

        def run_window():
            stats = capi.FrameStats()
            for k, (arr, n) in enumerate(ecalls):
                st = integrate_n(hptr, arr, n, 1, ctypes.byref(stats) if k == len(ecalls) - 1 else None)  # D2H of the result
                if st != 0:
                    raise RuntimeError(f"kb_integrate_frames (host) failed: {st}")
            h.synchronize()
        # untimed pass first (staging buffers), on other stamps: reuse the same frames with later stamps is not possible
        # (stamps must increase), so the window is timed on first use after one small warm-up call
        barrier()
        t0 = time.perf_counter()
        run_window()
        dt_local = time.perf_counter() - t0
        t = torch.tensor([dt_local, float(len(need))], device=dev, dtype=torch.float64)
        all_t = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(all_t, t)
        dt_max = max(float(x[0].item()) for x in all_t)
        deliveries = sum(float(x[1].item()) for x in all_t)
        e2e = {"value": n_e / dt_max, "unit": "frames/s", "h2d_bytes_per_step": int(deliveries * P * bpp),
               "d2h_bytes_per_step": world * (ctypes.sizeof(capi.FrameStats) + 64), "frames_per_step": n_e,
               "note": "every rank integrates the frames that touch its cells from its own pinned host buffers "
                       "(kb_integrate_frames, KB_MEM_HOST_ASYNC, %d frames/call) over its own PCIe link; max over ranks" % B}

    if rank == 0:
        A = np.array([x.cpu().numpy() for x in all_stats])
        parts = [[int(v) & ((1 << 64) - 1) for v in c.cpu().tolist()] for c in all_cs]
        fps = n_frames / (gpu_ms * 1e-3)
        full = [a.elapsed_time(b) / n_groups(n) for a, b, n in samples]
        n_calls = sum(n_groups(n) for s in range(Wm, Wm + K) for _, n in calls[s])
        roof = roofline_block(args, GROUP, n_calls, busy[0], float(np.mean(full) * 1e3) if full else None, nv, nsem, nblk,
                              my_frames, P, bpp, world=world)
        gbps = [float(A[r, 6] / (A[r, 5] * 1e-3) / 1e9) if A[r, 5] > 0 else 0.0 for r in range(world)]
        out = {
            "metric": "rgbd_frames_per_sec_integrated", "value": fps, "unit": "frames/s", "n_gpus": world,
            "steps": K, "warmup": Wm, "ms_per_step": gpu_ms / K, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload if not args.small else "hall160-small", "image": [W, H], "voxel_size": mc.voxel_size,
                       "voxels_per_side": 16, "truncation": mc.truncation_distance, "semantics": f"MLE L={L_LABELS}",
                       "frames_per_step": F, "frames_per_call": B, "frames_per_kernel_group": GROUP, "wire_format": "depth f32 + label i32 (8 B/px)", "lap_frames": lap,
                       "live_blocks_all_ranks": int(A[:, 7].sum()),
                       "l2": "inputs larger than L2: each step streams %.1f GB of frames" % (F * P * bpp / 1e9),
                       "parallelism": "cell shard x%d (%s); stream resident %s; every rank pulls the "
                                      "frames that touch its cells over NVLink (CUDA IPC peer mappings, transport: %s) and fuses them in stream order; "
                                      "no collective in the data path" % (world, layout_desc, {"striped": "striped over the ranks' pools (%d-frame chunks, round robin)" % stripe,
                                                                                "routed": "in the ranks' pools, every %d-frame chunk on a rank whose cells it touches (pose-aware ingest)" % stripe,
                                                                                "rank0": "on rank 0"}[args.ingest], args.gather),
                       "layout_max_frames_per_rank": layout_proxy, "render_s": round(t_render, 1)},
            "per_frame": {"voxels_updated": float(A[:, 0].sum()) / n_frames, "voxels_semantic": float(A[:, 1].sum()) / n_frames,
                          "blocks_visited": float(A[:, 2].sum()) / n_frames, "frame_deliveries": float(A[:, 3].sum()) / n_frames},
            "shards": {"frames_per_rank": [int(x) for x in A[:, 3]], "remote_frames_per_rank": [int(x) for x in A[:, 4]],
                       "busy_ms_per_rank": [round(x, 2) for x in busy], "blocks_per_rank": [int(x) for x in A[:, 7]]},
            "exchange": {"kind": "one-sided NVLink pull (kb_gather_run), overlapped with the previous step's fusion",
                         "bytes_pulled_all_ranks": float(A[:, 6].sum()), "gbps_per_rank": [round(x, 1) for x in gbps],
                         "gather_ms_per_rank": [round(float(x), 2) for x in A[:, 5]],
                         "reference_gbps": 770.0, "reference": "measured peer copy per direction (B200_PROFILING.md)"},
            "checksum": combine_checksums(parts),
            "roofline": roof, "cpu_baseline": None, "e2e": e2e, "gpu_launches": 6 * n_calls, "clocks": clocks, "wall_s_timed": wall,
        }
        emit(out)
    dist.barrier()
    for s in gplans:
        lib.kb_gather_plan_destroy(gplans[s])
    h.close()
    for r_ in rx:
        r_.close()
    pool.close()
    return None


def main():
    args = parse_args()
    quiet_stdout()
    if args.dump_outputs and (args.impl != "b200" or args.workload == "dynamic" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        raise SystemExit("bench.py: --dump-outputs covers the single-GPU hall workloads (--impl b200, 1 GPU, not --workload dynamic)")
    if args.impl == "reference":
        return main_reference(args)
    if args.workload == "dynamic":
        if int(os.environ.get("WORLD_SIZE", "1")) > 1:
            return main_dynamic_sharded(args)
        return main_dynamic(args)

    import torch
    import torch.distributed as dist
    import khronos_b200 as kb
    from khronos_b200 import capi, synthetic as syn

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    shard_note = None
    if world > 1 and args.shard == "cells":
        shard_note = main_hall_cells(args, world, rank, local_rank, dev)
        if shard_note is None:
            dist.destroy_process_group()
            return
        # peer memory unavailable on this box: fall back to the round-1 design (hash shard + NCCL broadcast)
    F, K, Wm = args.frames_per_step, args.steps, args.warmup
    if args.small:
        F = min(F, 64)
        args.lap_frames = min(args.lap_frames, 256)

    # nvidia-smi needs a few hundred ms to start and the timed region is short: start it now (it samples through
    # rendering and warm-up; only the samples inside the timed window are reported)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    cam, scene, poses, stamps = workload(args)
    lap = len(poses)
    P = cam.width * cam.height
    # ---- inputs into HBM (rank 0 renders; N>1: other ranks receive each step's frames by broadcast)
    t_render = time.perf_counter()
    if rank == 0:
        depth, label = syn.render_stream(scene, cam, poses, stamps, device=dev, dtype=torch.float32)
    else:
        depth = label = None
    compact = args.wire == "compact"
    f32u8 = args.wire == "f32u8"
    if f32u8 and world == 1:
        raise SystemExit("--wire f32u8 only changes what is broadcast: use it with --gpus N > 1 (torchrun)")
    bpp = 3 if compact else (5 if f32u8 else BYTES_PER_PIXEL_IN)
    if compact and rank == 0:
        # sensor-native formats: 16-bit millimetres (values < 32768, so int16 storage is bit-identical to u16), u8 ids
        depth = (depth * 1000.0).round().to(torch.int16)
        label = label.to(torch.uint8)
    torch.cuda.synchronize()
    t_render = time.perf_counter() - t_render
    if world > 1 and compact:
        HW = cam.height * cam.width
        rxp = [torch.empty((F, 3 * HW), dtype=torch.uint8, device=dev) for _ in range(2)]
        rx = [(b[:, :2 * HW].view(torch.int16).view(F, cam.height, cam.width), b[:, 2 * HW:].view(F, cam.height, cam.width)) for b in rxp]
    elif world > 1 and f32u8:
        # lossless narrow wire: depth stays f32, the (< 256) label ids travel as u8; the receiving ranks' frames carry
        # kb_frame.depth + kb_frame.label_u8 and the library widens the labels on the device
        HW = cam.height * cam.width
        rxp = [torch.empty((F, 5 * HW), dtype=torch.uint8, device=dev) for _ in range(2)]
        rx = [(b[:, :4 * HW].view(torch.float32).view(F, cam.height, cam.width), b[:, 4 * HW:].view(F, cam.height, cam.width)) for b in rxp]
    elif world > 1:
        # one packed receive buffer per step: [F, 2, H, W] int32 = (depth bits, label) -> a single broadcast
        rxp = [torch.empty((F, 2, cam.height, cam.width), dtype=torch.int32, device=dev) for _ in range(2)]
        rx = [(b[:, 0].view(torch.float32), b[:, 1]) for b in rxp]

    mm_hdl, tx = None, None
    if world > 1 and args.bcast == "multimem":
        # receive buffers from symmetric memory (same layout as above) + a local transmit buffer on the ingest rank
        import torch.distributed._symmetric_memory as symm_mem
        shape, dt = rxp[0].shape, rxp[0].dtype
        rxp, mm_hdl = [], []
        for _ in range(2):
            t = symm_mem.empty(int(np.prod(shape)), dtype=dt, device=dev)
            mm_hdl.append(symm_mem.rendezvous(t, dist.group.WORLD))
            rxp.append(t.view(shape))
        if not mm_hdl[0].multicast_ptr:  # 0 when the system has no NVLS multicast support
            raise SystemExit("--bcast multimem: no NVLS multicast mapping for the symmetric buffer on this system")
        HW = cam.height * cam.width
        if compact:
            rx = [(b[:, :2 * HW].view(torch.int16).view(F, cam.height, cam.width), b[:, 2 * HW:].view(F, cam.height, cam.width)) for b in rxp]
        elif f32u8:
            rx = [(b[:, :4 * HW].view(torch.float32).view(F, cam.height, cam.width), b[:, 4 * HW:].view(F, cam.height, cam.width)) for b in rxp]
        else:
            rx = [(b[:, 0].view(torch.float32), b[:, 1]) for b in rxp]
        if rank == 0:
            tx = torch.empty(shape, dtype=dt, device=dev)
            if compact:
                txv = (tx[:, :2 * HW].view(torch.int16).view(F, cam.height, cam.width), tx[:, 2 * HW:].view(F, cam.height, cam.width))
            elif f32u8:
                txv = (tx[:, :4 * HW].view(torch.float32).view(F, cam.height, cam.width), tx[:, 4 * HW:].view(F, cam.height, cam.width))
            else:
                txv = (tx[:, 0].view(torch.float32), tx[:, 1])
        mcopy = kb.lib().kb_multicast_copy
        mcopy.restype = ctypes.c_int

    mc, ic = map_configs(args)
    h = kb.create_map(mc, ic, capi.default_tracking_config(), None, device=local_rank)
    h.set_camera(cam)
    if args.no_cull:
        h.set_culling(False)
    if world > 1:
        h.set_shard(rank, world)
    stream = torch.cuda.Stream(device=dev)
    h.set_stream(stream.cuda_stream)

    def frame_index(step, j):
        return (step * F + j) % lap

    def stamp_of(step, j):
        g = step * F + j
        return 1_000_000_000 + g * 33_333_333

    B = F if args.batch <= 0 else max(1, min(args.batch, F))  # frames per kb_integrate_frames call
    integrate_n = h._fn("integrate_frames")
    hptr = h._h

    def make_step_batches(step, dbuf, lbuf, base):
        """ctypes Frame arrays (one per kb_integrate_frames call) for one step; images at frame offset
        base+j of (dbuf, lbuf), or at the lap index when base is None."""
        out = []
        for j0 in range(0, F, B):
            fr = []
            for j in range(j0, min(j0 + B, F)):
                i = frame_index(step, j)
                k = i if base is None else base + j
                if compact:
                    fr.append(h.make_frame(None, poses[i], stamp_of(step, j), depth_u16=dbuf[k].data_ptr(),
                                           label_u8=lbuf[k].data_ptr(), memory=capi.MEM_DEVICE))
                elif f32u8:
                    fr.append(h.make_frame(dbuf[k].data_ptr(), poses[i], stamp_of(step, j), label_u8=lbuf[k].data_ptr(),
                                           memory=capi.MEM_DEVICE))
                else:
                    fr.append(h.make_frame(dbuf[k].data_ptr(), poses[i], stamp_of(step, j), label=lbuf[k].data_ptr(),
                                           memory=capi.MEM_DEVICE))
            arr = (capi.Frame * len(fr))(*fr)
            out.append((arr, len(fr)))
        return out

    # frame descriptors are built outside the timed region (they only hold pointers, poses, stamps)
    if world > 1:
        prebuilt = {s: make_step_batches(s, rx[s % 2][0], rx[s % 2][1], 0) for s in range(Wm + K)}
    else:
        prebuilt = {s: make_step_batches(s, depth, label, None) for s in range(Wm + K)}

    buf_free = [torch.cuda.Event(), torch.cuda.Event()] if world > 1 else None  # rx[b] no longer read by kernels

    def run_step(step, sample_events=None):
        if world > 1:
            # double-buffered: the broadcast of step s+1 (torch's stream) overlaps the fusion of step s
            # (the handle's stream); rx[b] is overwritten only after the kernels of step s-2 are done
            bsel = step % 2
            db, lb = rx[bsel]
            cur = torch.cuda.current_stream()
            cur.wait_event(buf_free[bsel])
            if mm_hdl is not None:
                # NVLS: every rank has released rx[bsel] (barrier), rank 0 stores the step's frames once to the multicast
                # address, a second barrier publishes them
                mm_hdl[bsel].barrier()
                if rank == 0:
                    idx = torch.tensor([frame_index(step, j) for j in range(F)], device=dev)
                    txv[0].copy_(depth.index_select(0, idx))
                    txv[1].copy_(label.index_select(0, idx))
                    nbytes = tx.numel() * tx.element_size()
                    st = mcopy(ctypes.c_void_p(int(mm_hdl[bsel].multicast_ptr)), ctypes.c_void_p(tx.data_ptr()),
                               ctypes.c_size_t(nbytes - nbytes % 16), ctypes.c_void_p(cur.cuda_stream))
                    if st != 0:
                        raise RuntimeError(f"kb_multicast_copy failed: {st}")
                    if nbytes % 16:  # tail (never for the shapes used here)
                        rxp[bsel].view(-1).view(torch.uint8)[nbytes - nbytes % 16:].copy_(tx.view(-1).view(torch.uint8)[nbytes - nbytes % 16:])
                mm_hdl[bsel].barrier()
            else:
                if rank == 0:
                    idx = torch.tensor([frame_index(step, j) for j in range(F)], device=dev)
                    db.copy_(depth.index_select(0, idx))
                    lb.copy_(label.index_select(0, idx))
                dist.broadcast(rxp[bsel], 0)
            stream.wait_stream(cur)
        with torch.cuda.stream(stream):
            for j, (arr, n) in enumerate(prebuilt[step]):
                if sample_events is not None and n >= GROUP:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    st = integrate_n(hptr, arr, n, 1, None)
                    e1.record(stream)
                    sample_events.append((e0, e1, n))
                else:
                    st = integrate_n(hptr, arr, n, 1, None)
                if st != 0:
                    raise RuntimeError(f"kb_integrate_frames failed: {st}")
            if world > 1:
                buf_free[step % 2].record(stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for s in range(Wm):
        run_step(s)
    barrier()
    t64_0 = h.get_totals64()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    samples = []
    wall0 = time.perf_counter()
    ev0.record(stream)
    for s in range(Wm, Wm + K):
        run_step(s, samples)
    ev1.record(stream)
    barrier()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop(wall0, wall0 + wall) if rank == 0 else None
    gpu_ms = ev0.elapsed_time(ev1)
    if world > 1:
        # the device-timed region excludes nothing: broadcasts run on torch's stream between the
        # recorded events' stream work, so use the barrier-bracketed wall time, max over ranks
        t = torch.tensor([wall * 1e3], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        gpu_ms = float(t.item())
    t64_1 = h.get_totals64()
    if t64_1.capacity_exceeded:
        raise SystemExit("bench.py: block pool exhausted (capacity_exceeded): results incomplete")
    # order-independent checksum of the map after the timed region (same value for every --gpus N: the bench verifies itself)
    cs = h.map_checksum()
    if args.dump_outputs:  # before the e2e windows and legs below, which integrate more frames into this map
        dump_outputs(h, args.dump_outputs)
    pairs = t64_1.block_frame_pairs - t64_0.block_frame_pairs
    n_frames = K * F
    # 64-bit cumulative counters (kb_get_totals64): the 32-bit ones wrap after ~36 k frames of this workload
    nv = t64_1.voxels_updated - t64_0.voxels_updated
    nsem = t64_1.voxels_semantic - t64_0.voxels_semantic
    nblk = t64_1.blocks_in_frustum - t64_0.blocks_in_frustum
    if world > 1:
        t = torch.tensor([nv, nsem, nblk], device=dev, dtype=torch.float64)
        dist.all_reduce(t)
        nv_all, nsem_all, nblk_all = [float(x) for x in t.tolist()]
        cst = torch.tensor([int(c) - (1 << 64) if int(c) >= (1 << 63) else int(c) for c in cs], device=dev, dtype=torch.int64)
        all_cs = [torch.empty_like(cst) for _ in range(world)]
        dist.all_gather(all_cs, cst)
        cs_parts = [[int(v) & ((1 << 64) - 1) for v in c.cpu().tolist()] for c in all_cs]
    else:
        nv_all, nsem_all, nblk_all = float(nv), float(nsem), float(nblk)
        cs_parts = [cs]
    fps = n_frames / (gpu_ms * 1e-3)
    full = [a.elapsed_time(b) / n_groups(n) for a, b, n in samples]
    kern_us = float(np.mean(full) * 1e3) if full else None  # main-stream time per 32-frame kernel group, from per-call events
    n_launch = sum(n_groups(n) for s in range(Wm, Wm + K) for _, n in prebuilt[s])
    roof = roofline_block(args, GROUP, n_launch, gpu_ms, kern_us, nv, nsem, nblk, n_frames, P, bpp, world=world)

    # ---- secondary legs (N = 1): output tick on the benchmarked map (after the checksum: it integrates more frames)
    legs = {}
    if world == 1 and not args.no_legs and not compact and args.workload == "hall640":
        import bench_legs
        tick_step = Wm + K  # stamps after the timed steps and before the e2e windows (stamps must not decrease)

        def tick_batch(t):
            fr = [h.make_frame(depth[(t * 12 + j) % lap].data_ptr(), poses[(t * 12 + j) % lap], stamp_of(tick_step, t * 12 + j),
                               label=label[(t * 12 + j) % lap].data_ptr(), memory=capi.MEM_DEVICE) for j in range(12)]
            return (capi.Frame * 12)(*fr), 12
        try:
            legs["output_tick"] = bench_legs.leg_output_tick(h, tick_batch)
        except Exception as e:  # noqa: BLE001 - a failing leg must not take the headline down; it is reported
            legs["output_tick"] = {"error": str(e)[:300]}

    # ---- e2e: host (pinned) images through the same C ABI, H2D inside the timed region (rank-local)
    e2e = None
    if not args.no_e2e and world == 1:
        n_e = min(args.e2e_frames, lap)

        def host_window(step, as_compact):
            """Pinned host copies of the n_e frames that follow `step`, plus the kb_integrate_frames calls."""
            idx = [frame_index(step, j) for j in range(n_e)]
            it = torch.tensor(idx, device=dev)
            dsel, lsel = depth.index_select(0, it), label.index_select(0, it)
            if as_compact and not compact:  # quantise the f32 pool to the sensor-native formats for this window
                dsel, lsel = (dsel * 1000.0).round().to(torch.int16), lsel.to(torch.uint8)
            hd = torch.empty(dsel.shape, dtype=dsel.dtype, pin_memory=True)
            hl = torch.empty(lsel.shape, dtype=lsel.dtype, pin_memory=True)
            hd.copy_(dsel)
            hl.copy_(lsel)
            torch.cuda.synchronize()
            if as_compact:
                fr = [h.make_frame(None, poses[idx[j]], stamp_of(step, j), depth_u16=hd[j].data_ptr(), label_u8=hl[j].data_ptr(),
                                   memory=capi.MEM_HOST_ASYNC) for j in range(n_e)]
            else:
                fr = [h.make_frame(hd[j].data_ptr(), poses[idx[j]], stamp_of(step, j), label=hl[j].data_ptr(),
                                   memory=capi.MEM_HOST_ASYNC) for j in range(n_e)]
            calls = [((capi.Frame * len(fr[j0:j0 + B]))(*fr[j0:j0 + B]), len(fr[j0:j0 + B])) for j0 in range(0, n_e, B)]
            return calls, (hd, hl)

        def run_window(calls):
            stats = capi.FrameStats()
            for j, (arr, n) in enumerate(calls):
                last = j == len(calls) - 1
                st = integrate_n(hptr, arr, n, 1, ctypes.byref(stats) if last else None)  # D2H of the result
                if st != 0:
                    raise RuntimeError(f"kb_integrate_frames (host) failed: {st}")
            h.synchronize()

        def timed_window(step, as_compact):
            calls, keep = host_window(step, as_compact)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run_window(calls)
            return time.perf_counter() - t0

        timed_window(Wm + K + 1, compact)        # untimed: the library allocates its staging buffers here
        dt = timed_window(Wm + K + 2, compact)
        e2e = {"value": n_e / dt, "unit": "frames/s", "h2d_bytes_per_step": n_e * P * bpp,
               "d2h_bytes_per_step": ctypes.sizeof(capi.FrameStats) + 64, "frames_per_step": n_e,
               "note": "host pinned depth+label ring -> kb_integrate_frames(KB_MEM_HOST_ASYNC, %d frames/call); stats read back at step end" % B}
        if not compact:
            # informational: the same window shipped in the sensor-native compact formats (kb_frame.depth_u16 / label_u8)
            timed_window(Wm + K + 3, True)
            dtc = timed_window(Wm + K + 4, True)
            e2e["compact_wire"] = {"value": n_e / dtc, "unit": "frames/s", "h2d_bytes_per_step": n_e * P * 3,
                                   "note": "u16 millimetre depth + u8 labels, expanded on the device (3 B/pixel over PCIe)"}

        # ---- the same window as a Khronos run sees it: an output tick every 12 frames (min_output_separation 0.4 s of a 30 Hz
        # stream, uHumans2.yaml:38; ActiveWindow::extractOutputData, active_window.cpp:217-249): mesh of the updated blocks
        # (kb_generate_mesh + kb_get_mesh: the tick's device->host traffic) and the clearUpdated loop (:169-171)
        try:
            step_t = Wm + K + 5
            idx = [frame_index(step_t, j) for j in range(n_e)]
            it = torch.tensor(idx, device=dev)
            hd = torch.empty((n_e, cam.height, cam.width), dtype=torch.float32, pin_memory=True)
            hl = torch.empty((n_e, cam.height, cam.width), dtype=torch.int32, pin_memory=True)
            hd.copy_(depth.index_select(0, it) if not compact else depth.index_select(0, it).float() * 0.001)
            hl.copy_(label.index_select(0, it).to(torch.int32))
            torch.cuda.synchronize()
            fr = [h.make_frame(hd[j].data_ptr(), poses[idx[j]], stamp_of(step_t, j), label=hl[j].data_ptr(), memory=capi.MEM_HOST_ASYNC)
                  for j in range(n_e)]
            tcalls = [((capi.Frame * len(fr[j0:j0 + 12]))(*fr[j0:j0 + 12]), len(fr[j0:j0 + 12])) for j0 in range(0, n_e, 12)]
            h.generate_mesh(True, True)
            h.clear_updated()
            gen, getm = h._fn("generate_mesh"), h._fn("get_mesh")
            cap_v = 4_000_000
            pts, col, lab = np.empty((cap_v, 3), np.float32), np.empty((cap_v, 3), np.uint8), np.empty(cap_v, np.uint32)
            bi, off = np.empty((8192, 3), np.int32), np.empty(8193, np.int64)
            d2h = 0
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for arr, n in tcalls:
                st = integrate_n(hptr, arr, n, 1, None)
                if st != 0:
                    raise RuntimeError(f"kb_integrate_frames (host) failed: {st}")
                nb_, nv_ = ctypes.c_int32(0), ctypes.c_int64(0)
                h._check(gen(hptr, 1, 1, ctypes.c_float(1e-4), ctypes.byref(nb_), ctypes.byref(nv_)))
                if nv_.value > cap_v or nb_.value > 8192:
                    raise RuntimeError("mesh tick larger than the bench buffers")
                h._check(getm(hptr, ctypes.c_void_p(bi.ctypes.data), ctypes.c_void_p(off.ctypes.data), ctypes.c_void_p(pts.ctypes.data),
                              ctypes.c_void_p(col.ctypes.data), ctypes.c_void_p(lab.ctypes.data), ctypes.c_int64(cap_v)))
                h.clear_updated()
                d2h += nv_.value * 19 + nb_.value * 20 + 8
            h.synchronize()
            dtt = time.perf_counter() - t0
            e2e["with_output_ticks"] = {"value": n_e / dtt, "unit": "frames/s", "ticks": len(tcalls), "h2d_bytes_per_step": n_e * P * 8,
                                        "d2h_bytes_per_step": int(d2h),
                                        "note": "host pinned frames in calls of 12 (one output period), after each: marching cubes on the device + "
                                                "triangles to the host + clearUpdated — the per-frame and per-tick work of ActiveWindow that this "
                                                "library replaces, end to end"}
        except Exception as e:  # noqa: BLE001 - informational block; it must not take the headline down
            e2e["with_output_ticks"] = {"error": str(e)[:200]}

    # ---- CPU baseline on a bounded sample of the same stream (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n_c = min(args.cpu_sample_frames, lap) if not args.small else min(96, lap)

        def host_chunk(i, k):  # the CPU arm gets the same frames (compact: expanded the same way, float(u16) * 0.001f)
            d, l = depth[i:i + k].cpu().numpy(), label[i:i + k].cpu().numpy()
            if compact:
                d, l = d.astype(np.float32) * np.float32(0.001), l.astype(np.int32)
            return d, l

        probe = host_chunk(0, 12)
        nt = best_cpu_threads(args, cam, probe, poses, list(range(12)))
        cfps, cores, secs, n_done = run_cpu_stream(args, cam, host_chunk, poses, stamps, n_c, args.cpu_sample_seconds, threads=nt)
        cpu = {"value": cfps, "unit": "frames/s", "cores": cores, "kind": "port",
               "sample": f"first {n_done} frames of the lap into an empty map, oracle port, {secs:.1f} s of integration, "
                         f"best of a thread-count sweep up to {os.cpu_count()} host threads"}

    if world == 1 and not args.no_legs and not compact and args.workload == "hall640":
        import bench_legs
        nt_legs = locals().get("nt") or min(32, os.cpu_count() or 1)
        for name, fn in (("dynamic", lambda: bench_legs.leg_dynamic_hall(args, cam, scene, poses, stamps, depth, label, dev, nt_legs,
                                                                           n_timed=600 if not args.small else 24, small=args.small)),
                         ("next_rows", lambda: bench_legs.leg_next_rows(dev, small=args.small, cpu=not args.no_cpu_baseline))):
            try:
                legs[name] = fn()
            except Exception as e:  # noqa: BLE001
                legs[name] = {"error": str(e)[:300]}

    if rank == 0:
        total = h.get_totals()
        out = {
            "metric": "rgbd_frames_per_sec_integrated", "value": fps, "unit": "frames/s", "n_gpus": world,
            "steps": K, "warmup": Wm, "ms_per_step": gpu_ms / K, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload if not args.small else "hall160-small",
                       "image": [cam.width, cam.height], "voxel_size": mc.voxel_size, "voxels_per_side": 16,
                       "truncation": mc.truncation_distance, "semantics": f"MLE L={L_LABELS}", "frames_per_step": F, "frames_per_call": B,
                       "frames_per_kernel_group": GROUP,
                       "wire_format": ("depth u16 mm + label u8 (3 B/px), expanded on device" if compact else
                                       "depth f32 + label u8 (5 B/px, lossless; labels widened on device)" if f32u8 else
                                       "depth f32 + label i32 (8 B/px)"),
                       "lap_frames": lap, "live_blocks_rank0": total.total_blocks,
                       "l2": "inputs larger than L2: each step streams %.1f GB of frames" % (F * P * bpp / 1e9),
                       "parallelism": ("block-hash shard x%d, %s frame broadcast%s" % (world, "NVLS multimem" if args.bcast == "multimem" else "NCCL",
                                                                                   (" (fallback: " + shard_note + ")") if shard_note else "")) if world > 1 else "single GPU",
                       "render_s": round(t_render, 1)},
            "per_frame": {"voxels_updated": nv_all / n_frames, "voxels_semantic": nsem_all / n_frames,
                          "blocks_visited": nblk_all / n_frames,
                          "block_frame_pairs_after_k0_culling_rank0": pairs / n_frames},
            "checksum": combine_checksums(cs_parts),
            "roofline": roof,
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": 6 * n_launch, "clocks": clocks,
            "wall_s_timed": wall,
        }
        if legs:
            out["configs"] = {"dynamic": legs.get("dynamic")}
            out["output_tick"] = legs.get("output_tick")
            out["next_rows"] = legs.get("next_rows")
        emit(out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
