#!/usr/bin/env python
"""bench.py -- frames/s of the dense tracking-and-fusion hot path on B200 (BASELINE.json metric).

Workload (N=1): BASELINE.json configs[1] -- synthetic 640x480 RGB-D stream into a 512^3 TSDF volume (6 m), ICP-only
tracker {10,5,4} iterations, volume shifting on (-t 14, overlap 2).  A "step" is ONE frame through
KintinuousTracker::processFrame's replacement (kt_process_frame*): pyramid -> 19 ICP iterations -> shift test ->
integrate -> raycast + model pyramid.

  value : frames/s with the RGB-D frames already resident in HBM (kt_process_frame_device), whole job (all ranks).
  e2e   : frames/s through the public C ABI with HOST (pinned) buffers: H2D of depth + rgb and D2H of the pose are
          inside the timed region (kt_process_frame).
  roofline / stages : CUDA-event stage timers of the tracker (on its own stream), algorithmic bytes from DESIGN.md section 4.
  cpu_baseline : the CPU oracle ("port") on a bounded sample of the same workload, on this box's host cores.
  --impl reference : the reference's OWN CUDA kernels (oracle/_ref/libkt_ref_512.so, compiled from /root/reference with
          two mechanical patches), driven by the restated host loop with the reference's launch / sync pattern.
          The reference has no CPU implementation of this path; if the library is missing, the CPU oracle port is timed.
Timing: W>=3 warm-up frames, exactly K timed frames between barrier + cuda synchronize, max over ranks, CUDA clocks sampled
with nvidia-smi during the timed region.  Inputs: 96 distinct frames (147 MB) cycled, i.e. larger than the 126 MB L2.
Multi-GPU (torchrun): the headline line is weak scaling -- rank r tracks its own stream into its own volume (independent sessions, no
data-path collective).  At every N the same JSON line carries a `zslab` sub-record: ONE stream fused into ONE 1024^3 volume shared by all
N GPUs (BASELINE configs[3]; replicated TSDF with owner P2P stores, block-cyclic colour planes, banded ray cast with the model-map
all-gather as P2P stores; DESIGN.md section 6) -- strong scaling of one stream; --mode zslab runs the main legs in that mode instead.
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

ROWS, COLS, VOL, SIZE = 480, 640, 512, 6.0
N_INPUT_FRAMES = int(os.environ.get("KT_BENCH_FRAMES", "96"))
P_LEVELS = [ROWS * COLS >> (2 * l) for l in range(4)]
ICP_ITERS = [10, 5, 4, 0]
TRACKER_NAMES = {0: "ICP-only tracker", 1: "RGB-D-only tracker (-r)", 2: "ICP+RGB-D tracker (-ri)"}
METRIC_TAGS = {0: "ICP-only", 1: "RGB-D-only", 2: "ICP+RGB-D"}


def _render_one(k):
    from kintinuous_b200 import synth
    return synth.render(k, COLS, ROWS)


def make_stream(n, offset=0, world=1, rank=0):
    """n frames of the synthetic trajectory, played forward then backward (ping-pong) so any number of steps is continuous.
    Under torchrun rank 0 renders once into /dev/shm and the other ranks load it (they all need the same frames)."""
    cache = f"/dev/shm/kt_bench_frames_{n}_{offset}_{COLS}x{ROWS}.npz"
    if world > 1:
        import torch.distributed as dist
        if rank == 0 and not os.path.exists(cache):
            fr = make_stream(n, offset)
            np.savez(cache + ".tmp.npz", depth=np.stack([f[0] for f in fr]), rgb=np.stack([f[1] for f in fr]))
            os.replace(cache + ".tmp.npz", cache)
        dist.barrier()
        z = np.load(cache)
        return [(np.ascontiguousarray(z["depth"][i]), np.ascontiguousarray(z["rgb"][i])) for i in range(n)]
    ks = [offset + i for i in range(n)]
    try:
        from concurrent.futures import ProcessPoolExecutor
        with ProcessPoolExecutor(max_workers=min(16, os.cpu_count() or 1)) as ex:
            frames = list(ex.map(_render_one, ks, chunksize=2))
    except Exception:
        frames = [_render_one(k) for k in ks]
    return frames


def pingpong(i, n):
    period = 2 * (n - 1)
    j = i % period
    return j if j < n else period - j


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region.  NVML in-process (initialised before the warm-up, polled every 10 ms by
    a thread): spawning `nvidia-smi` at the start of a 70 ms timed region perturbed the region itself (its start-up takes driver
    locks; observed as an occasional 2x slower device leg).  Falls back to an `nvidia-smi -lms` child started early if NVML is absent."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None
        self.h = None
        self.run = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None
            q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
            try:
                self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(index), "-lms", "100"],
                                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
                self.t = threading.Thread(target=self._read_smi, daemon=True); self.t.start()
            except Exception:
                self.proc = None

    def _read_smi(self):
        for line in self.proc.stdout:
            if self.run:
                self.rows.append([x.strip() for x in line.split(",")])

    def _poll(self):
        nv = self.nv
        while self.run:
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.rows.append((mhz, mask))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        self.run = True
        if self.h is not None:
            self.t = threading.Thread(target=self._poll, daemon=True); self.t.start()

    def stop(self):
        self.run = False
        if self.h is not None:
            self.t.join(timeout=1.0)
            sm = [r[0] for r in self.rows]
            reasons = sorted({name for r in self.rows for bit, name in self.REASONS.items() if r[1] & bit})
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(sm), "source": "nvml, 2 ms poll"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml and nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm), "source": "nvidia-smi -lms 100"}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def dist_setup(n_gpus, init=True):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and init:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl" if not os.environ.get("KT_BENCH_GLOO") else "gloo")
    return world, rank, local


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()


def max_over_ranks(x, world, device):
    if world == 1:
        return x
    import torch, torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def cpu_baseline_leg(frames, n_sample):
    """CPU oracle port on a bounded sample (rank 0 only)."""
    from oracle import refbind
    import kintinuous_b200 as kb
    o = refbind.CpuOracle()
    cores = o.lib.ktoracle_hardware_threads() or (os.cpu_count() or 1)
    o.lib.ktoracle_set_threads(cores)
    cfg = kb.Config.default(rows=ROWS, cols=COLS, vol=VOL, odometry=0)
    t = o.tracker(refbind.TrackerConfig.from_kt(cfg))
    n_sample = min(n_sample, len(frames) - 1)
    t.process(frames[0][0], frames[0][1], 0)          # first frame (no odometry) is not timed
    t0 = time.time()
    for k in range(1, 1 + n_sample):
        t.process(frames[k][0], frames[k][1], k)
    dt = time.time() - t0
    t.close()
    return {"value": n_sample / dt, "unit": "frames/s", "cores": int(cores), "kind": "port",
            "sample": f"{n_sample} frames of the same 640x480 -> 512^3 ICP workload, oracle/kt_oracle_cpu.cpp on {cores} std::threads ({dt:.1f} s)"}


def shared_volume_leg(kb, torch, args, world, rank, local, device, dev_depth, dev_rgb, n, warmup):
    """One RGB-D stream fused into ONE volume (BASELINE configs[3]: 1024^3) by all `world` GPUs: TSDF replicated (owner stores changed
    voxels into every replica over NVLink from inside integrate_kernel), colour / weight planes block-cyclic, ray casting split into
    image bands with the model-map all-gather as P2P stores in the kernel epilogue, ICP replicated; no collective library call on the
    data path.  Strong scaling of one stream: frames/s of THE stream, max over ranks, CUDA events on the tracker stream."""
    V = args.shared_vol
    cfg = kb.Config.default(rows=ROWS, cols=COLS, vol=V, odometry=args.odometry, device=local, rank=rank if world > 1 else 0, world=world)
    trk = kb.Tracker(cfg)
    if world > 1:
        from kintinuous_b200 import mgpu
        mgpu.connect(trk)
    steps = args.steps
    prewarm = 40

    def run(k, i):
        for _ in range(k):
            j = pingpong(i, n); jn = pingpong(i + 1, n)
            trk.process_frame_device(dev_depth[j], dev_rgb[j], i)
            if not args.no_prefetch:
                trk.prefetch_frame(dev_depth[jn], dev_rgb[jn])
            i += 1
        return i
    i = run(prewarm + warmup + 1, 0)
    torch.cuda.synchronize(); barrier(world)
    trk.span_mark(0)
    i = run(steps, i)
    trk.span_mark(1)
    dt = trk.span_elapsed_ms() * 1e-3
    torch.cuda.synchronize(); barrier(world)
    dt = max_over_ranks(dt, world, device)
    trk.set_stage_timing(True)
    acc = np.zeros(6); kacc = np.zeros(3); m = 0
    for _ in range(12):
        j = pingpong(i, n); p = trk.process_frame_device(dev_depth[j], dev_rgb[j], i); i += 1
        if p.shifted == 0:
            acc += np.array(trk.stage_ms()); kacc += np.array(trk.kernel_ms()); m += 1
    st = (acc / max(1, m)).tolist(); kst = (kacc / max(1, m)).tolist()
    info = trk.mgpu_info()
    trk.close()
    barrier(world)
    P0 = ROWS * COLS
    maps_bytes = sum((P0 >> (2 * l)) * 24 for l in range(4)) + P0 * 4
    return {"value": steps / dt, "unit": "frames/s", "n_gpus": world, "vol": V, "steps": steps, "ms_per_step": 1e3 * dt / steps, "scaling": "strong",
            "workload": f"ONE synthetic {COLS}x{ROWS} RGB-D stream into ONE {V}^3 volume (6 m) shared by {world} GPU(s), {TRACKER_NAMES[args.odometry]}",
            "parallelism": ("single GPU" if world == 1 else
                            f"TSDF plane replicated on {world} GPUs (owner stores changed voxels into every replica: NVLink P2P stores inside integrate_kernel), colour/weight planes block-cyclic "
                            f"(blocks of {info['block']} storage z planes), ray cast split into {world} image bands with the model-map all-gather as P2P stores in the kernel epilogue, "
                            "flag barriers in peer memory, ICP replicated; no NCCL call on the data path"),
            "stages_ms_rank0": {nm: st[k] for k, nm in enumerate(["pyramid", "odometry", "shift", "integrate", "raycast"])},
            "kernels_ms_rank0": {"icp": kst[0], "ztable+integrate": kst[1], "raycast": kst[2],
                                 "note": "the launches alone; the stage timers above include the cross-GPU barriers, i.e. the wait for the slowest rank"},
            "p2p_model_map_bytes_per_frame": int(maps_bytes * (world - 1)) if world > 1 else 0,
            "arena_mb_per_gpu": info["arena_mb"]}


def run_reference(args, world, rank, local):
    """--impl reference: the reference's own CUDA kernels behind the restated host loop (rank 0 only)."""
    if rank != 0:
        return
    from oracle import refbind
    import kintinuous_b200 as kb
    cfg = kb.Config.default(rows=ROWS, cols=COLS, vol=args.vol, odometry=args.odometry)
    n_frames = N_INPUT_FRAMES                         # the same frame set as the b200 arm (same_config)
    frames = make_stream(n_frames)
    PREWARM = int(os.environ.get("KT_BENCH_PREWARM", "150"))
    warmup = max(3, args.warmup)
    # n_gpus is what this arm USED: the reference has no multi-GPU path, rank 0 runs it on one GPU whatever --gpus says
    line = {"metric": f"frames/s {COLS}x{ROWS} into {args.vol}^3 TSDF ({METRIC_TAGS[args.odometry]} tracker)", "unit": "frames/s", "n_gpus": 1, "requested_gpus": args.gpus, "steps": args.steps, "warmup": warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": f"synthetic {COLS}x{ROWS} RGB-D stream, {args.vol}^3 volume (6 m), {TRACKER_NAMES[args.odometry]} {{10,5,4}}, shifting on (-t 14)", "frames_cycled": n_frames,
                       "prewarm_frames": PREWARM, "untimed_frames_before_region": PREWARM + warmup + 1}}
    use_cuda = False
    try:
        import torch
        use_cuda = torch.cuda.is_available() and refbind.RefCuda.available(args.vol)
    except Exception:
        use_cuda = False
    if use_cuda:
        import torch
        torch.cuda.set_device(0)
        ref = refbind.RefCuda(args.vol)
        t = ref.tracker(refbind.TrackerConfig.from_kt(cfg))
        sync = torch.cuda.synchronize
        kind, cores = "reference", 1
        sample = "every step: the reference's own CUDA kernels (oracle/_ref/libkt_ref_<vol>.so = /root/reference src/frontend/cuda/*.cu recompiled for sm_100) on cuda:0, original launch shapes and 26 syncs/frame, restated host loop on 1 host thread, blocking H2D from pageable memory"
    else:
        o = refbind.CpuOracle()
        cores = o.lib.ktoracle_hardware_threads() or 1
        o.lib.ktoracle_set_threads(cores)
        t = o.tracker(refbind.TrackerConfig.from_kt(cfg))
        sync = lambda: None
        kind = "port"
        sample = f"oracle/_ref unavailable: CPU oracle port on {cores} threads"
        args.steps = min(args.steps, 8); warmup = 1; PREWARM = 0
        line["steps"], line["warmup"] = args.steps, warmup
        line["config"]["prewarm_frames"] = 0; line["config"]["untimed_frames_before_region"] = 2
    i = 0
    for _ in range(PREWARM + warmup + 1):             # the same untimed lead-in as the b200 arm (GPU clocks, allocator, first shifts)
        d, c = frames[pingpong(i, n_frames)]; t.process(d, c, i); i += 1
    sync(); t0 = time.perf_counter()
    for _ in range(args.steps):
        d, c = frames[pingpong(i, n_frames)]; t.process(d, c, i); i += 1
    sync(); dt = time.perf_counter() - t0
    v = args.steps / dt
    line.update({"value": v, "ms_per_step": 1e3 * dt / args.steps,
                 "cpu_baseline": {"value": v, "unit": "frames/s", "cores": int(cores), "kind": kind, "sample": sample},
                 "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    print(json.dumps(line), flush=True)


DUMP_LIMIT_BYTES = 64_000_000        # everything --dump-outputs writes, all files together
DUMP_MAP_PIXELS = 640 * 480          # a larger frame's model maps are dumped at a fixed, seeded sample of this many pixels
DUMP_VOXELS = 2_000_000


def _map_with_mask(m):
    """A vertex / normal map (x, y, z planes first) as the reference stores it marks a pixel without a surface with NaN in its x plane
    (its y / z planes keep stale values).  Dumped as the map with those pixels zeroed in all three planes plus a 0 / 1 mask of the
    valid pixels, so every value is finite and two runs compare element for element."""
    valid = ~np.isnan(m[0])
    m = np.where(valid[None], m, np.float32(0)).astype(np.float32)
    return m, valid.astype(np.float32)


def dump_outputs(out_dir, trk, pose, zslab):
    """What the timed path computed in its last step, as float32 / float64 .npy files of at most DUMP_LIMIT_BYTES together (about 26 MB
    at 640x480): the pose that kt_process_frame_device returned, the model vertex / normal maps the frame left for the next one (with
    their validity masks), and the TSDF value and weight of a fixed, seeded sample of voxels.  The samples are drawn with seed 0 from
    the frame size and the volume side alone, so every run with the same arguments dumps the same pixels and voxels.  In the z-slab
    mode rank 0 holds only its own storage planes of the volume, so the voxels are drawn from those (Tracker.export_owned)."""
    R, t, global_t, wrap = pose.as_tuple()
    out = {"pose_R": R, "pose_t": t, "pose_global_t": global_t, "pose_voxel_wrap": wrap.astype(np.float64)}
    npix = trk.cfg.rows * trk.cfg.cols
    pix = np.sort(np.random.default_rng(0).choice(npix, DUMP_MAP_PIXELS, replace=False)) if npix > DUMP_MAP_PIXELS else None
    for name, which in (("model_vmap", 2), ("model_nmap", 3)):
        m = trk.download_map(which, 0)
        if pix is not None:
            m = m.reshape(3, -1)[:, pix]
        out[name], out[name + "_valid"] = _map_with_mask(m)
    tsdf, color = trk.export_owned() if zslab else trk.export_volume()
    idx = np.sort(np.random.default_rng(0).choice(tsdf.size, min(DUMP_VOXELS, tsdf.size), replace=False))
    out["volume_sample_tsdf"] = tsdf.reshape(-1)[idx].astype(np.float32)
    out["volume_sample_weight"] = color.reshape(-1, 4)[idx, 3].astype(np.float32)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    for name, a in out.items():
        if not np.isfinite(a).all():
            raise RuntimeError(f"--dump-outputs: {name} is not finite")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="streams", choices=["streams", "zslab"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample", type=int, default=48)
    ap.add_argument("--no-prefetch", action="store_true", help="do not give the kt_prefetch_frame hint (A/B)")
    ap.add_argument("--no-shared-volume", action="store_true", help="skip the extra one-stream / one-shared-1024^3-volume leg (the zslab sub-record)")
    ap.add_argument("--shared-vol", type=int, default=1024)
    ap.add_argument("--shared-only", action="store_true", help="diagnostic: run only the shared-volume leg and print its record")
    ap.add_argument("--vol", type=int, default=VOL)
    ap.add_argument("--scale", type=int, default=1, help="image scale: 1 = 640x480 (configs 1-3), 2 = 1280x960 (configs[4])")
    ap.add_argument("--odometry", type=int, default=0, help="0 ICP (configs[1]), 2 ICP+RGB-D (configs[2])")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed device path computed in its last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.shared_only or args.impl == "reference"):
        ap.error("--dump-outputs dumps the b200 arm's main timed path; it does not apply with --shared-only or --impl reference")
    global ROWS, COLS, P_LEVELS, N_INPUT_FRAMES
    if args.scale != 1:
        ROWS, COLS = 480 * args.scale, 640 * args.scale
        P_LEVELS = [ROWS * COLS >> (2 * l) for l in range(4)]
        N_INPUT_FRAMES = max(8, N_INPUT_FRAMES // (args.scale * args.scale))      # same bytes of distinct input
    if args.impl == "reference":                      # rank 0 alone runs it; no process group, no collective
        world, rank, local = dist_setup(args.gpus, init=False)
        run_reference(args, world, rank, local)
        return
    world, rank, local = dist_setup(args.gpus)

    import torch
    import kintinuous_b200 as kb
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- kintinuous_b200 has no CPU path (use --impl reference for the CPU/legacy arm)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    warmup = max(3, args.warmup)
    PREWARM = int(os.environ.get("KT_BENCH_PREWARM", "150"))

    frames = make_stream(N_INPUT_FRAMES, offset=0, world=world, rank=rank)
    n = len(frames)
    # resident inputs (value) and pinned host inputs (e2e)
    dev_depth = [torch.from_numpy(f[0].view(np.int16)).to(device) for f in frames]
    dev_rgb = [torch.from_numpy(f[1]).to(device) for f in frames]
    pin_depth = [torch.from_numpy(f[0].view(np.int16)).pin_memory() for f in frames]
    pin_rgb = [torch.from_numpy(f[1]).pin_memory() for f in frames]
    if args.shared_only:
        rec = shared_volume_leg(kb, torch, args, world, rank, local, device, dev_depth, dev_rgb, n, warmup)
        if world > 1:
            import torch.distributed as dist
            dist.barrier(); dist.destroy_process_group()
        if rank == 0:
            print(json.dumps({"zslab": rec}), flush=True)
        return
    zslab = (args.mode == "zslab" and world > 1)
    cfg = kb.Config.default(rows=ROWS, cols=COLS, vol=args.vol, odometry=args.odometry, device=local,
                            rank=rank if zslab else 0, world=world if zslab else 1)

    def run(tracker, use_host, steps, start):
        """Process `steps` frames from frame index `start`; returns the next index and the pose of the last frame."""
        i = start
        p = None
        for _ in range(steps):
            j = pingpong(i, n)
            jn = pingpong(i + 1, n)
            # kt_prefetch_frame (public API hint): the next frame's copy and pose-independent front end overlap this frame's fusion
            if use_host:
                p = tracker.process_frame(pin_depth[j].data_ptr(), pin_rgb[j].data_ptr(), i)
                if not args.no_prefetch:
                    tracker.prefetch_frame(pin_depth[jn].data_ptr(), pin_rgb[jn].data_ptr())
            else:
                p = tracker.process_frame_device(dev_depth[j], dev_rgb[j], i)
                if not args.no_prefetch:
                    tracker.prefetch_frame(dev_depth[jn], dev_rgb[jn])
            i += 1
        return i, p

    results = {}
    clocks = None
    for leg in ("device", "host"):
        trk = kb.Tracker(cfg)
        if zslab:
            from kintinuous_b200 import mgpu
            mgpu.connect(trk)
        sampler = ClockSampler(local) if (leg == "device" and rank == 0) else None      # NVML init / child start-up outside the timed region
        # frame 0 + W warm-up frames as the contract asks, preceded by PREWARM more untimed frames: the inputs were rendered on the CPU
        # for seconds with the GPU idle, and W = 3 frames (1 ms) do not bring its clocks and the allocator to steady state
        i, _ = run(trk, leg == "host", PREWARM + warmup + 1, 0)
        torch.cuda.synchronize(); barrier(world)
        if leg == "device" and rank == 0:
            sampler.start()
        l0 = trk.launch_count()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        trk.span_mark(0)                                    # CUDA events on the tracker's own stream (torch events would not see it)
        i, last = run(trk, leg == "host", args.steps, i)
        trk.span_mark(1)
        dt = trk.span_elapsed_ms() * 1e-3                   # synchronises on the closing event
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        l1 = trk.launch_count()
        barrier(world)
        if leg == "device" and rank == 0:
            clocks = sampler.stop()
        if dt <= 0:
            raise RuntimeError("device stopwatch failed")
        dt = max_over_ranks(dt, world, device)
        results[leg] = {"dt": dt, "wall": max_over_ranks(wall, world, device), "launches": l1 - l0}
        if leg == "device" and args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, trk, last, zslab)
        if leg == "device":
            # stage timers (CUDA events on the tracker's stream) over a few extra frames, outside the timed region
            trk.set_stage_timing(True)
            acc = np.zeros(6)
            m = 0
            icp_ms = 0.0
            for _ in range(16):
                j = pingpong(i, n); p = trk.process_frame_device(dev_depth[j], dev_rgb[j], i); i += 1
                ms = np.array(trk.stage_ms())
                if p.shifted == 0:
                    acc += ms; m += 1; icp_ms += trk.icp_kernel_ms()
            results["stages_ms"] = (acc / max(1, m)).tolist()
            results["icp_kernel_ms"] = icp_ms / max(1, m)
        trk.close()

    # ---- BASELINE configs[3]: ONE stream into ONE 1024^3 volume shared by all `world` GPUs (the north_star's multi-GPU design): a
    # sub-record of the same JSON line at every N (N = 1: the single-GPU figure it is compared with) ----
    shared = None
    if args.mode == "streams" and not args.no_shared_volume and args.scale == 1:
        try:
            shared = shared_volume_leg(kb, torch, args, world, rank, local, device, dev_depth, dev_rgb, n, warmup)
        except Exception as e:  # the headline number must survive a failure of the extra leg
            shared = {"value": None, "error": str(e)[:300]}
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    peak, peak_src = measured_peak()
    st = results["stages_ms"]
    names = ["pyramid", "odometry", "shift", "integrate", "raycast"]
    # algorithmic bytes per pixel and Gauss-Newton iteration (DESIGN.md section 4): ICP 48 B (two float3 current maps + two float3
    # model maps), photometric 14 B (last/next depth 4+4, last/next intensity 1+1, next gradients 2+2)
    per_px = {0: 48, 1: 14, 2: 62}[args.odometry]
    icp_bytes = sum(per_px * P_LEVELS[l] * ICP_ITERS[l] for l in range(4))
    tracker_name = TRACKER_NAMES[args.odometry]
    kernel_name = ("icp_frame_kernel (1 cooperative launch per frame = 19 Gauss-Newton iterations, TMA-staged current maps, FP64 solve on device)"
                   if args.odometry == 0 else
                   "rgbd_frame_kernel (1 cooperative launch per frame = 19 iterations of photometric" + (" + point-to-plane" if args.odometry == 2 else "") + " Gauss-Newton, FP64 solve on device)")
    alg_bytes = {"pyramid": 4 * P_LEVELS[0] + sum(2 * P_LEVELS[l] + 2 * P_LEVELS[l + 1] for l in range(3)) + sum(2 * P_LEVELS[l] + 24 * P_LEVELS[l] for l in range(4)),
                 "odometry": icp_bytes, "integrate": None, "raycast": None}
    stages = {nm: {"ms": st[k]} for k, nm in enumerate(names)}
    for nm in ("pyramid", "odometry"):
        stages[nm]["alg_bytes"] = alg_bytes[nm]
        stages[nm]["gbs"] = alg_bytes[nm] / (st[names.index(nm)] * 1e-3) / 1e9 if st[names.index(nm)] > 0 else None
    dom = max(names, key=lambda nm: st[names.index(nm)])
    # dominant kernel = icp_frame_kernel: ONE launch per frame that runs all 19 Gauss-Newton iterations (48 B per pixel and iteration,
    # DESIGN.md section 4); duration from CUDA events recorded around that launch on the tracker's stream
    icp_ms = results.get("icp_kernel_ms", 0.0) or st[1]
    ach = icp_bytes / (icp_ms * 1e-3) / 1e9 if icp_ms > 0 else None
    traffic = None
    traffic_file = None
    try:                                                      # dram__bytes_read.sum + dram__bytes_write.sum of the committed ncu capture
        import csv, glob
        kname = "icp_frame_kernel" if args.odometry == 0 else "rgbd_frame_kernel"
        cands = sorted(glob.glob(os.path.join(ROOT, "profiles", f"r2_ncu_full_*{kname}*.csv"))) or sorted(glob.glob(os.path.join(ROOT, "profiles", f"r1_ncu_full_v10_{kname}.csv")))
        traffic_file = os.path.relpath(cands[-1], ROOT)
        rows = list(csv.reader(open(cands[-1])))
        H, U, Vv = rows[0], rows[1], rows[2]
        def val(name):
            i = H.index(name); x = float(Vv[i]); u = U[i].lower()
            return x * (1e6 if u.startswith("mbyte") else 1e3 if u.startswith("kbyte") else 1e9 if u.startswith("gbyte") else 1.0)
        traffic = val("dram__bytes_read.sum") + val("dram__bytes_write.sum")
    except Exception:
        traffic = None
    # compulsory DRAM bytes of the launch: the four map sets of the levels in use, read once (48 B/pixel; later iterations hit L2 / smem)
    compulsory = sum(per_px * P_LEVELS[l] for l in range(4) if ICP_ITERS[l] > 0)
    roofline = {"kernel": kernel_name, "bound": "hbm",
                "achieved": ach, "peak": peak, "unit": "GB/s", "frac": (ach / peak) if ach else None, "traffic": traffic,
                "traffic_source": f"ncu --set full capture {traffic_file} (dram__bytes_read.sum + dram__bytes_write.sum, one launch); not re-measured in this run" if traffic else None,
                "compulsory_dram_bytes": compulsory, "frac_compulsory_dram": (compulsory / (icp_ms * 1e-3) / 1e9 / peak) if icp_ms > 0 else None,
                "peak_source": peak_src, "bytes_per_launch": icp_bytes, "avg_launch_ms": icp_ms,
                "note": "algorithmic bytes / CUDA-event time of that launch; the kernel is latency-bound by design at 640x480 (19 sequential reduce+solve steps, each a grid-wide exchange; inputs L2- / shared-memory-resident so DRAM traffic equals one compulsory read of the maps, far below the algorithmic bytes); see DESIGN.md section 4 and profiles/r2_ncu_summary.md",
                "dominant_stage": dom}
    dt = results["device"]["dt"]
    streams = 1 if zslab else world          # z-slab: all ranks work on ONE stream (strong scaling)
    value = streams * args.steps / dt
    e2e_v = streams * args.steps / results["host"]["dt"]
    line = {"metric": f"frames/s {COLS}x{ROWS} into {args.vol}^3 TSDF ({METRIC_TAGS[args.odometry]} tracker)", "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "ms_per_step": 1e3 * dt / args.steps, "wall_ms_per_step": 1e3 * results["device"]["wall"] / args.steps, "timing": "CUDA events on the tracker stream, max over ranks", "higher_is_better": True, "scaling": "strong" if zslab else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"synthetic {COLS}x{ROWS} RGB-D stream, {args.vol}^3 volume (6 m), {tracker_name} {{10,5,4}}, shifting on (-t 14)", "parallelism": (f"one stream, volume z-slab sharded over {world} GPUs (P2P raycast, replicated ICP)" if zslab else f"{world} independent streams"), "vol": args.vol, "odometry": args.odometry,
                       "prewarm_frames": PREWARM, "untimed_frames_before_region": PREWARM + warmup + 1, "prefetch_hint": not args.no_prefetch, "l2": f"inputs larger than L2: {n} frames x {ROWS * COLS * 5 / 1e6:.2f} MB = {n * ROWS * COLS * 5 / 1e6:.0f} MB cycled (ping-pong)"},
            "e2e": {"value": e2e_v, "unit": "frames/s", "h2d_bytes_per_step": ROWS * COLS * 5, "d2h_bytes_per_step": 48},
            "gpu_launches": int(results["device"]["launches"]), "clocks": clocks, "roofline": roofline, "stages": stages}
    if shared is not None:
        line["zslab"] = shared
    if not args.no_cpu_baseline:
        try:
            line["cpu_baseline"] = cpu_baseline_leg(frames, args.cpu_sample)
        except Exception as e:  # the oracle is a checker, its absence must not hide the GPU number
            line["cpu_baseline"] = {"value": None, "unit": "frames/s", "cores": 0, "kind": "port", "sample": f"unavailable: {e}"}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
