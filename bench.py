#!/usr/bin/env python
"""bench.py — PointFusion frames/sec (640x480, B=8 sequences of L=32 frames per GPU, odom='gt', fwd only).

    python bench.py [--gpus N --steps K --warmup W]            our CUDA arm
    python bench.py ... --dump-outputs DIR                     also write the last timed step's result to DIR/*.npy
    python bench.py --impl reference [...]                     the CPU oracle port timed on the host cores
    torchrun ... bench.py --gpus N ...                         one rank per GPU (weak scaling: B=8 per GPU)

One "step" = one whole `PointFusion(odom='gt')(frames)` call over a (B, L) batch of synthetic RGB-D
sequences = B*L frame updates (per frame: K1r frame records, K2/K3 project+select, K3c per-tile append counts,
K4 merge+append).  The timed region is EXACTLY --steps steps; with `--repeats R` it is measured R times back to back
(default 1) and the MEDIAN region is reported (all of them are listed under "timed_regions_ms").  The inputs are
seeded, so the same arguments give the same inputs on every run; --dump-outputs writes what the timed path returned
in its last step, so that two builds can be compared output for output.
Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for what each key means.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # NCCL's version banner must not land on stdout (ONE JSON line)

METRIC = "PointFusion frames/sec (640x480, B=8)"
UNIT = "frames/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="gsx", choices=["gsx", "reference"])
    ap.add_argument("--batch", type=int, default=8, help="sequences per GPU")
    ap.add_argument("--seqlen", type=int, default=32)
    ap.add_argument("--height", type=int, default=480)
    ap.add_argument("--width", type=int, default=640)
    ap.add_argument("--cpu-sample-frames", type=int, default=12, help="frames of the CPU-baseline sample (B=1)")
    ap.add_argument("--repeats", type=int, default=1, help="timed regions of --steps steps each")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's poses, map sizes and a fixed sample of map rows as DIR/*.npy")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra-configs", action="store_true", help="skip the B=1 / L=32 (config 2) line")
    ap.add_argument("--no-icp", action="store_true", help="skip the secondary ICP-odometry measurement")
    ap.add_argument("--no-raw", action="store_true", help="skip the dataset-native (uint8/uint16) ingest measurement")
    ap.add_argument("--no-e2e", action="store_true", help="diagnostic runs only: skip the end-to-end leg (e2e = null)")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms",
                 "25"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
_BEST_THREADS = {}


def best_thread_count(H, W):
    """The reference's op chain (dominated by torch.unique(dim=0)) does not scale with threads, and on a
    100+-core host it is SLOWER with every core than with a few.  Give the baseline its best case: try a few
    thread counts on a 3-frame sample and keep the fastest."""
    import torch

    key = (H, W)
    if key not in _BEST_THREADS:
        cores = os.cpu_count() or 1
        best = None
        for t in sorted(set(min(cores, c) for c in (4, 8, 16, 32, cores))):
            torch.set_num_threads(t)
            fps = cpu_reference_run(1, 3, H, W, threads=t)[0]
            if best is None or fps > best[0]:
                best = (fps, t)
        _BEST_THREADS[key] = best[1]
    return _BEST_THREADS[key]


def cpu_reference_run(frames_B, frames_L, H, W, seed=0, threads=None):
    """Times the CPU oracle port (torch-CPU restatement of the reference's op chain) on the host cores."""
    import torch

    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import gsx_oracle as oracle
    from gradslam_b200.synthetic import make_sequence

    cores = threads if threads is not None else best_thread_count(H, W)
    torch.set_num_threads(cores)
    rgb, depth, K, poses = make_sequence(frames_B, frames_L, H, W, seed=seed)
    t0 = time.perf_counter()
    res = oracle.run_slam(rgb, depth, K, poses, odom="gt")
    dt = time.perf_counter() - t0
    return frames_B * frames_L / dt, dt, cores, res.map.counts()


def run_reference(args, rank, world):
    if rank != 0:
        return
    sample_B, sample_L = 1, args.cpu_sample_frames
    # warm-up steps run a shorter sample; every timed step is the same bounded sample of the workload
    best_thread_count(args.height, args.width)  # doubles as warm-up
    # keep the whole arm within ~2 minutes whatever --steps is: shrink the per-step sample if needed
    _, dt4, _, _ = cpu_reference_run(1, 4, args.height, args.width)
    budget_frames = int(120.0 / max(1, args.steps) / max(dt4 / 4.0, 1e-3))
    sample_L = max(2, min(sample_L, budget_frames))
    vals = []
    for _ in range(max(1, args.steps)):
        fps, dt, cores, _ = cpu_reference_run(sample_B, sample_L, args.height, args.width)
        vals.append((fps, dt))
    fps = sum(v[0] for v in vals) / len(vals)
    ms = 1e3 * sum(v[1] for v in vals) / len(vals)
    sample = ("PointFusion(odom=gt) %dx%d B=%d sequence x L=%d frames per step: a bounded sample of the B=%d x L=%d "
              "workload (the CPU arm runs ~2 frames/s), timed with the thread count that is fastest for this op chain "
              "(%d of %d cores; torch.unique(dim=0) dominates and slows down with more threads)" % (
                  args.width, args.height, sample_B, sample_L, args.batch, args.seqlen, cores, os.cpu_count() or 1))
    cfg = workload_config(args, 1)
    # say what RAN: the sampled batch / length, not the workload it was sampled from
    cfg.update({"workload": cfg["workload"].split(", %dx%d" % (args.width, args.height))[0] +
                ", %dx%d, B=%d sequence x L=%d frames per step (bounded sample of B=%d x L=%d)" % (
                    args.width, args.height, sample_B, sample_L, args.batch, args.seqlen),
                "global_batch": sample_B, "seq_len": sample_L, "frames_per_step": sample_B * sample_L,
                "parallelism": "host cores (%d threads)" % cores,
                "sampled_from": {"global_batch": args.batch, "seq_len": args.seqlen}})
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# GSX_BENCH_EXCHANGE: diagnostic only.  overlap (default, the product path): the maps of step k travel while step k+1 is
# fused;  serial: exchange, then the next step;  none: no exchange (NOT the metric - the line says so in config).
EXCHANGE_SCHEDULE = os.environ.get("GSX_BENCH_EXCHANGE", "overlap")


def workload_config(args, world):
    return {
        "workload": "PointFusion(odom='gt', dist_th=0.05, angle_th=20, sigma=0.6) forward over synthetic box-room "
                    "RGB-D sequences, %dx%d, B=%d sequences x L=%d frames per GPU" % (
                        args.width, args.height, args.batch, args.seqlen),
        "global_batch": args.batch * world, "seq_len": args.seqlen, "height": args.height, "width": args.width,
        "frames_per_step": args.batch * world * args.seqlen, "parallelism": "batch-sharded x%d" % world,
        "map_exchange": None if world == 1 else "%s (%s)" % (
            {2: "peer pulls over CUDA IPC, job-wide store"}.get(world, "NCCL all-gather of the packed row arrays")
            if os.environ.get("GSX_MAP_EXCHANGE", "auto") == "auto" else os.environ["GSX_MAP_EXCHANGE"],
            EXCHANGE_SCHEDULE),
        "l2_policy": "inputs (%.0f MB depth+rgb per GPU per step) exceed the 126 MB L2" % (
            args.batch * args.seqlen * args.height * args.width * 16 / 1e6),
    }


DUMP_BYTES = 48 << 20  # budget of the sampled map rows in --dump-outputs


def dump_outputs(out_dir, pc, poses):
    """Writes one PointFusion result as float32 / float64 .npy files: the recovered poses, the map sizes and the map's
    points, normals, colours and confidence counts at a fixed, seeded sample of row indices (map_rows.npy; rows past an
    element's size are zero).  The whole map (~140 MB at the default workload) is sampled to stay within DUMP_BYTES."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    B, n = pc.points_padded.shape[:2]
    keep = min(n, DUMP_BYTES // (max(B, 1) * 10 * 4))
    rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
    idx = rows.to(pc.points_padded.device)
    arrays = {"poses": poses, "num_points": pc.num_points_per_pointcloud.double(), "map_rows": rows.double(),
              "points": pc.points_padded[:, idx], "normals": pc.normals_padded[:, idx],
              "colors": pc.colors_padded[:, idx], "features": pc.features_padded[:, idx]}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().cpu().numpy())


# ------------------------------------------------------------------------------------------------------
def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    import gradslam_b200 as gs
    from gradslam_b200 import parallel, profiling
    from gradslam_b200.synthetic import make_sequence

    assert torch.cuda.is_available(), "bench.py (impl gsx) needs a GPU; there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # host buffers of this rank in the memory of its GPU's NUMA node (matters for the e2e leg at N > 1)
    host_cpus = parallel.bind_host_to_gpu(dev) if world > 1 else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner on stdout when the communicator is created; stdout must carry exactly
        # one JSON line, so point fd 1 at stderr until the first collective has gone through.
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)

    B, L, H, W = args.batch, args.seqlen, args.height, args.width
    rgb_h, depth_h, K_h, poses_h = make_sequence(B, L, H, W, seed=rank, pin_memory=True)
    K_h, poses_h = K_h.pin_memory(), poses_h.pin_memory()
    rgb_d, depth_d, K_d, poses_d = (t.to(dev) for t in (rgb_h, depth_h, K_h, poses_h))
    frames_dev = gs.RGBDImages(rgb_d, depth_d, K_d, poses_d)
    frames_host = gs.RGBDImages(rgb_h, depth_h, K_h, poses_h)
    slam = gs.PointFusion(odom="gt", device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    dl_stream = torch.cuda.Stream(device=dev)
    dl_state = {"host": None, "bytes": 0}

    def read_back(pc, poses, fused):
        """Result read-back of one step: recovered poses, map sizes and the fused map itself (packed rows, exact sizes)
        into pinned host memory, on a side stream so that it overlaps the next step's upload and fusion.  `fused`: event
        recorded when that step's fusion had been enqueued (the copies wait for it, not for the step enqueued since)."""
        dl_stream.wait_event(fused)
        if dl_state.get("poses") is None:
            dl_state["poses"] = torch.empty(poses.shape, dtype=poses.dtype, pin_memory=True)
        with torch.cuda.stream(dl_stream):
            dl_state["poses"].copy_(poses, non_blocking=True)
        poses.record_stream(dl_stream)
        host = pc.download(out=dl_state["host"], stream=dl_stream)
        dl_state["host"] = host
        rows = sum(host._host_counts())
        dl_state["bytes"] = rows * (32 + 16) + poses.numel() * 4 + len(host) * 8
        return dl_state["poses"], host

    # N > 1: two job-wide stores used alternately; each rank fuses its sequences straight into its block of one of them
    # and pulls the peers' rows into the other blocks (GSX_BENCH_STORE=fresh: a fresh local map and a fresh gathered
    # store per step, own rows copied - the round-1 behaviour, for comparison)
    stores = []
    exchange = parallel.exchange_mode(dev) if world > 1 else None
    if world > 1 and os.environ.get("GSX_BENCH_STORE", "shared" if exchange == "peer" else "fresh") == "shared":
        stores = [parallel.GatheredMaps(B, L * H * W, dev) for _ in range(2)]

    def run_steps(frames, steps, d2h):
        """`steps` whole-batch PointFusion calls.  N>1: the final-map exchange of step k (communication stream) overlaps
        the fusion of step k+1; the last one is awaited before returning.  d2h: the result (poses + the fused map of this
        rank) is read back to pinned host memory; the read-back of step k overlaps step k+1."""
        res = None
        pending = None  # (gather handle, poses) of the previous step
        prev = None  # (map, poses) of the previous step, still to be read back
        for i in range(steps):
            store = stores[i % len(stores)] if stores else None
            if store is not None:
                # the block is reused every other step: wait (on the device) for its last exchange and read-back
                torch.cuda.current_stream(dev).wait_stream(dl_stream)
                pc, poses = slam(frames, out=store.reset())
            else:
                pc, poses = slam(frames)
            fused = torch.cuda.Event()
            fused.record()
            if pending is not None:  # step k-1's maps travel while step k (just enqueued) computes
                parallel.gather_maps_end(pending[0], wait=False)
            if d2h and prev is not None:
                res = read_back(*prev)
            if world > 1 and EXCHANGE_SCHEDULE == "serial":  # diagnostic: the exchange alone on the GPU, then the next step
                parallel.gather_maps(pc, into=store)
            elif world > 1 and EXCHANGE_SCHEDULE != "none":
                pending = (parallel.gather_maps_begin(pc, into=store), poses)
            prev = (pc, poses, fused)
        if pending is not None:
            parallel.gather_maps_end(pending[0], wait=True)
        if d2h:
            res = read_back(*prev)
            torch.cuda.current_stream(dev).wait_stream(dl_stream)
            return res
        return prev[:2]  # (map, poses) of the last step, on the device

    def timed(frames, steps, d2h):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = run_steps(frames, steps, d2h)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms, res

    def timed_median(frames, steps, d2h, repeats):
        """`repeats` timed regions of exactly `steps` steps each; returns (median ms, all ms, last result)."""
        all_ms, res = [], None
        for _ in range(repeats):
            ms, res = timed(frames, steps, d2h)
            all_ms.append(ms)
        return sorted(all_ms)[len(all_ms) // 2], all_ms, res

    repeats = max(1, args.repeats)
    if world > 1:  # setup, not warm-up: let the caching allocator reach its steady state (two map stores and two sets
        run_steps(frames_dev, 3, d2h=False)  # of gather buffers are alive at once in the pipelined loop)
    run_steps(frames_dev, max(args.warmup, 3), d2h=False)  # same (pipelined) code path as the timed region
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_dev, all_dev, last = timed_median(frames_dev, args.steps, False, repeats)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)
    del last
    if args.no_e2e:
        ms_e2e, all_e2e = float("nan"), []
    else:
        run_steps(frames_host, 3, d2h=True)
        ms_e2e, all_e2e, res = timed_median(frames_host, args.steps, True, repeats)

    # extra: the same job fed in dataset-native form (uint8 colour + uint16 depth, 5 B/pixel over PCIe instead of 16)
    raw_extra = None
    if not args.no_raw:
        import numpy as np

        from gradslam_b200.ingest import RawRGBD

        col_u8 = torch.from_numpy((rgb_h.numpy() * 255.0).astype(np.uint8)).pin_memory()
        dep_u16 = torch.from_numpy(np.round(depth_h.numpy()[..., 0] * 5000.0).astype(np.uint16)).pin_memory()
        raw = RawRGBD(col_u8, dep_u16, K_h, poses_h, scaling_factor=5000.0)
        run_steps(raw, 3, d2h=True)
        ms_raw, _, _ = timed_median(raw, args.steps, True, min(repeats, 3))
        raw_extra = {"value": B * L * world * args.steps / (ms_raw / 1e3), "unit": UNIT, "ms_per_step": ms_raw / args.steps,
                     "h2d_bytes_per_step": col_u8.numel() + dep_u16.numel() * 2 + (K_h.numel() + poses_h.numel()) * 4,
                     "d2h_bytes_per_step": dl_state["bytes"],
                     "note": "PointFusion(odom='gt')(RawRGBD): uint8 colour + uint16 depth (TUM/ICL on-disk format, "
                             "depth = u16/5000) uploaded from pinned memory and converted on the device; same "
                             "read-back as e2e"}
        del raw, col_u8, dep_u16

    frames_per_step = B * L * world
    value = frames_per_step * args.steps / (ms_dev / 1e3)
    e2e = frames_per_step * args.steps / (ms_e2e / 1e3)
    h2d = (rgb_h.numel() + depth_h.numel() + K_h.numel() + poses_h.numel()) * 4
    d2h = dl_state["bytes"]

    # per-kernel timing + roofline of the dominant kernel (rank 0's GPU; every rank runs the same work)
    roofline, kernels, frames_info = None, None, None
    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        prof, frames_info = profiling.profile_pointfusion_gt(depth_d, rgb_d, K_d, poses_d, slam.dist_th, slam.dot_th,
                                                             slam.sigma)
        prof, frames_info = profiling.profile_pointfusion_gt(depth_d, rgb_d, K_d, poses_d, slam.dist_th, slam.dot_th,
                                                             slam.sigma)  # second pass = warm
        kernels = {}
        for name, rows in prof.items():
            tot_ms = sum(r[0] for r in rows)
            tot_b = sum(r[1] for r in rows)
            kernels[name] = {"launches": len(rows), "total_ms": tot_ms, "avg_us": 1e3 * tot_ms / max(1, len(rows)),
                             "algorithmic_GB_per_s": tot_b / max(tot_ms, 1e-9) / 1e6,
                             "algorithmic_MB_per_launch": tot_b / max(1, len(rows)) / 1e6}
        dom = max(kernels, key=lambda k: kernels[k]["total_ms"])
        ach = kernels[dom]["algorithmic_GB_per_s"]
        roofline = {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": None, "peak_source": peak_src,
                    "bytes_per_launch": kernels[dom]["algorithmic_MB_per_launch"] * 1e6,
                    "avg_launch_us": kernels[dom]["avg_us"]}
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tpath):  # dram bytes per launch from the committed ncu --set full capture
            roofline["traffic"] = json.load(open(tpath)).get(dom)

    # secondary measurement: the same PointFusion with its default ICP odometry (gradLM, 20 iterations, dsratio 4),
    # on a corner-facing variant of the scene (yaw0=0.6) where point-to-plane ICP is well conditioned; plus the
    # localisation call alone (K5 exact 1-NN + K6 rows / normal equations + K7 solve, 2 searches per iteration) with its
    # work in SURVEY.md §8(d)'s units and the CPU port of the same call beside it
    icp_extra = None
    if rank == 0 and not args.no_icp:
        from gradslam_b200.odometry.icputils import downsample_pointclouds, localize_against_map
        from gradslam_b200.slam.fusionutils import find_active_map_points

        Li, ds, iters = 8, 4, 20
        r2, d2, K2, p2 = make_sequence(B, Li, H, W, seed=100 + rank, yaw0=0.6)
        fr2 = gs.RGBDImages(r2.to(dev), d2.to(dev), K2.to(dev), p2.to(dev))
        slam2 = gs.PointFusion(odom="gradicp", device=dev)
        slam2(fr2)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            _, rec = slam2(fr2)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / 3
        icp_extra = {"workload": "PointFusion(odom='gradicp', numiters=20, dsratio=4) %dx%d B=%d L=%d, 1 GPU" % (W, H, B, Li),
                     "frames_per_s": B * Li / ms * 1e3, "ms_per_step": ms,
                     "max_abs_pose_error_vs_gt": float((rec.cpu() - p2).abs().max())}
        # the localisation of the last frame against the map of the first Li-1 frames, alone
        slam_gt = gs.PointFusion(odom="gt", device=dev)
        pc_map, _ = slam_gt(fr2[:, : Li - 1])
        live, prev = fr2[:, Li - 1], fr2[:, Li - 2]
        live.poses = prev.poses
        localize_against_map(pc_map, live, prev, ds, slam2.odomprov)
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(5):
            pose_dev = localize_against_map(pc_map, live, prev, ds, slam2.odomprov)
        e1.record()
        torch.cuda.synchronize(dev)
        ms_loc = e0.elapsed_time(e1) / 5
        ns = (d2[:, Li - 1, ::ds, ::ds, 0] > 0).flatten(1).sum(1).tolist()
        tgt = downsample_pointclouds(pc_map, find_active_map_points(pc_map, prev), ds)
        nt = [int(c) for c in tgt.num_points_per_pointcloud.tolist()]
        searches = 2 * iters
        flop = sum(a * b for a, b in zip(ns, nt)) * 8.0 * searches  # brute-force-equivalent pair evaluations
        k6_bytes = sum(ns) * 36.0 * searches
        icp_extra["localize"] = {
            "ms_per_call": ms_loc, "source_points": ns, "target_points": nt, "searches_per_call": searches,
            "K5_brute_force_equivalent_TFLOP_per_s": flop / (ms_loc * 1e-3) / 1e12,
            "K5_note": "SURVEY 8(d) unit: Ns*Nt pairs x 8 flop per search over the WHOLE call time (K5+K6+K7 and the two "
                       "gathers); targets > 4096 points are searched through an exact uniform grid (~1e2 distance "
                       "evaluations per query), so this is work AVOIDED, not FP32 throughput",
            "K6_algorithmic_GB_per_s": k6_bytes / (ms_loc * 1e-3) / 1e9,
            "K6_note": "36 B per source point per search (SURVEY 8(d)) over the whole call time: a lower bound",
        }
        if not args.no_cpu_baseline:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import gsx_oracle as oracle

            torch.set_num_threads(best_thread_count(H, W))
            ref_run = oracle.run_slam(r2[:1, : Li - 1], d2[:1, : Li - 1], K2[:1], p2[:1, : Li - 1], odom="gt")
            at_prev = oracle.frame_maps(d2[:1, Li - 1: Li], K2[:1], p2[:1, Li - 2: Li - 1])
            t0 = time.perf_counter()
            pose_cpu = oracle.odometry(ref_run.map, at_prev, p2[:1, Li - 2], K2[:1, 0], H, W, "gradicp", ds,
                                       dict(numiters=iters, damp=1e-8, dist_thresh=None, lambda_max=2.0, B=1.0, B2=1.0,
                                            nu=200.0))
            dt = time.perf_counter() - t0
            icp_extra["localize"]["cpu_port"] = {
                "seconds_per_call_B1": dt, "cores": os.cpu_count(),
                "kind": "oracle.odometry: torch-CPU restatement of ICPSLAM._localize with the brute-force KNN "
                        "restatement (oracle/knn1.c, OpenMP on all cores) in place of chamferdist",
                "gpu_over_cpu_per_sequence": dt / (ms_loc * 1e-3 / B),
                "max_abs_pose_diff_vs_cuda": float((pose_cpu[0] - pose_dev[0, 0].cpu()).abs().max())}

    # BASELINE.json configs[1]: one sequence (B=1), L=32, forward only - the launch-latency-bound end of the path
    small_extra = None
    if rank == 0 and not args.no_extra_configs:
        fr1 = gs.RGBDImages(rgb_d[:1], depth_d[:1], K_d[:1], poses_d[:1])
        for _ in range(3):
            slam(fr1)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            pc1, _ = slam(fr1)
        e1.record()
        torch.cuda.synchronize(dev)
        ms1 = e0.elapsed_time(e1) / 20
        small_extra = {"workload": "PointFusion(odom='gt') %dx%d B=1 L=%d, 1 GPU, forward (configs[1])" % (W, H, L),
                       "frames_per_s": L / ms1 * 1e3, "ms_per_step": ms1,
                       "us_per_frame": 1e3 * ms1 / L,
                       "vs_batched_per_frame": (ms1 / L) / ((ms_dev / args.steps) / (B * L))}

    # The other BASELINE.json configurations, so that they appear in a driver-run line (each guarded: a failure is
    # reported as {"error": ...} and never costs the headline).  configs[2]: ICPSLAM 640x480, 10 iterations, batch 8,
    # forward + backward; configs[3]: PointFusion 64-frame sequences, 4 per GPU (this GPU's share of the 32-sequence job);
    # configs[4]: PointFusion 1280x960, batch 8.
    other_configs = None
    if rank == 0 and world == 1 and not args.no_extra_configs:
        other_configs = {}

        def per_call_ms(fn, calls, warm=2):
            for _ in range(warm):
                fn()
            torch.cuda.synchronize(dev)
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(calls):
                fn()
            b_.record()
            torch.cuda.synchronize(dev)
            return a.elapsed_time(b_) / calls

        try:
            r3, d3, K3, p3 = make_sequence(B, 2, H, W, seed=0, yaw0=0.6)
            r3, K3 = r3.to(dev), K3.to(dev)
            d3g, p3g = d3.to(dev).requires_grad_(True), p3.to(dev).requires_grad_(True)
            icpslam = gs.ICPSLAM(odom="gradicp", numiters=10, dsratio=4, device=dev)
            fwd_ms = bwd_ms = 0.0
            calls = 5
            for it in range(2 + calls):
                d3g.grad = p3g.grad = None
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                ev[0].record()
                _, rec3 = icpslam(gs.RGBDImages(r3, d3g, K3, p3g))
                ev[1].record()
                rec3.sum().backward()
                ev[2].record()
                torch.cuda.synchronize(dev)
                if it >= 2:
                    fwd_ms += ev[0].elapsed_time(ev[1]) / calls
                    bwd_ms += ev[1].elapsed_time(ev[2]) / calls
            with torch.no_grad():
                fr3 = gs.RGBDImages(r3, d3g.detach(), K3, p3g.detach())
                fused_ms = per_call_ms(lambda: icpslam(fr3), calls)
                _, rec3f = icpslam(fr3)
            other_configs["config3_icpslam_fwd_bwd"] = {
                "workload": "ICPSLAM(odom='gradicp', numiters=10, dsratio=4) %dx%d B=%d L=2, inputs resident, "
                            "loss = poses.sum()" % (W, H, B),
                "forward_ms": fwd_ms, "backward_ms": bwd_ms, "fused_no_grad_forward_ms": fused_ms,
                "grads_finite": bool(torch.isfinite(d3g.grad).all() and torch.isfinite(p3g.grad).all()),
                "max_abs_pose_diff_fused_vs_differentiable": float((rec3f - rec3.detach()).abs().max()),
                "max_abs_pose_error_vs_gt": float((rec3.detach().cpu() - p3).abs().max())}
            del r3, d3, K3, p3, d3g, p3g, fr3, rec3, rec3f
        except Exception as exc:  # noqa: BLE001 - reported, not fatal
            other_configs["config3_icpslam_fwd_bwd"] = {"error": repr(exc)[:300]}
        for key, (Bc, Lc, Hc, Wc), what in (
                ("config4_b4_l64_per_gpu", (4, 64, H, W), "configs[3]: 64-frame sequences, 4 per GPU; each is two of the "
                 "bench's 32-frame trajectories through the same room back to back, i.e. the second half revisits"),
                ("config5_1280x960_b8", (8, 4, 960, 1280), "configs[4]: 1280x960, batch 8 (L=4)")):
            try:
                if key.startswith("config4") and B >= 8 and L * 2 == Lc:
                    half = B // 2
                    rc_, dc_, pc_ = (torch.cat([t[:half], t[half: 2 * half]], dim=1).contiguous()[:Bc]
                                     for t in (rgb_d, depth_d, poses_d))
                    Kc_ = K_d[:Bc].contiguous()
                else:
                    rc_, dc_, Kc_, pc_ = (t.to(dev) for t in make_sequence(Bc, Lc, Hc, Wc, seed=7))
                frc = gs.RGBDImages(rc_, dc_, Kc_, pc_)
                msc = per_call_ms(lambda: slam(frc), 5)
                other_configs[key] = {"workload": "PointFusion(odom='gt') %dx%d B=%d L=%d, 1 GPU, forward, inputs "
                                                  "resident (%s)" % (Wc, Hc, Bc, Lc, what),
                                      "frames_per_s": Bc * Lc / msc * 1e3, "ms_per_step": msc,
                                      "us_per_frame_per_sequence": 1e3 * msc / Lc}
                del rc_, dc_, Kc_, pc_, frc
            except Exception as exc:  # noqa: BLE001
                other_configs[key] = {"error": repr(exc)[:300]}
        torch.cuda.empty_cache()

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        fps, dt, cores, _ = cpu_reference_run(1, args.cpu_sample_frames, H, W)
        cpu_baseline = {"value": fps, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": "oracle.run_slam (torch-CPU restatement, torch.unique(dim=0) kept) PointFusion(odom=gt) "
                                  "%dx%d B=1 L=%d, %.1f s wall" % (W, H, args.cpu_sample_frames, dt)}

    if rank == 0:
        from gradslam_b200 import _C as _gsx
        groups = int(_gsx.lib().gsx_pointfusion_sequence_groups(B))
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, world),
            "e2e": None if args.no_e2e else {
                    "value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps,
                    "result": "poses + map sizes + the fused map of this rank (packed rows, exact sizes) into pinned "
                              "host memory, overlapped with the next step",
                    "host_cpus": host_cpus, "timed_regions_ms": all_e2e},
            # K1r + K2/K3 + K4 per frame and per concurrent batch group; K2 is skipped on the empty map
            "gpu_launches": groups * (3 * L - 1) * args.steps, "sequence_groups": groups,
            "repeats": repeats, "timed_regions_ms": all_dev,
            "roofline": roofline, "cpu_baseline": cpu_baseline, "clocks": clocks, "kernels": kernels,
            "icp_odometry": icp_extra, "e2e_raw_ingest": raw_extra, "config2_b1_l32": small_extra,
            "other_configs": other_configs,
            "final_map_points_per_sequence": (frames_info[-1]["map_points"] + frames_info[-1]["new"]) // B
            if frames_info else None,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
