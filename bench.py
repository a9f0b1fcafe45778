#!/usr/bin/env python
"""Headline benchmark: point-clouds/sec of the SECOND (SpMiddleFHD, KITTI-car grid) forward on synthetic 20k-point
clouds -- BASELINE.json `metric`, configs[1].

    python bench.py --gpus N --steps K --warmup W                 (N>1: launched under torchrun, one rank per GPU)
    python bench.py --config {second,pillars,cbgs} ...            (BASELINE configs[1] / [2] / [3] at their stated sizes)
    python bench.py --impl reference ...                          (the reference path on the host cores)
    python bench.py --dump-outputs DIR ...                        (also write the last timed step's detections to DIR)

One step = one pass of the whole hot path (voxelize -> reader -> sparse middle encoder -> RPN -> heads -> decode /
top-k / rotated NMS) over one batch of clouds per GPU.  The ranks' detections are exchanged with ONE all-gather after
the last step, inside the timed region, as the reference does (tools/dist_test.py:213-215).  Prints ONE JSON line.
"""
import argparse
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

N_CLOUD_POOL = 8       # distinct synthetic clouds cycled through the steps
WORKLOADS = {
    # name: (config file, points per cloud, point features, clouds per GPU per step, BASELINE.json config, head calibration)
    "second": dict(cfg="second_kitti_car.py", n_points=20000, ndim=4, batch=1, pass_fraction=0.03,
                   name="SECOND kitti_car_vfev3_spmiddlefhd_rpn1 forward, 20k synthetic pts"),
    "pillars": dict(cfg="pointpillars_kitti_car.py", n_points=20000, ndim=4, batch=8, pass_fraction=0.02,
                    name="PointPillars kitti_point_pillars_mghead forward, 20k synthetic pts"),
    "cbgs": dict(cfg="cbgs_nusc.py", n_points=35000, ndim=5, batch=4, pass_fraction=0.01,
                 name="CBGS nusc_all_vfev3_spmiddleresnetfhd_rpn2_mghead forward, 35k synthetic pts"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="det3d_b200", choices=["det3d_b200", "reference"])
    ap.add_argument("--config", default="second", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=None, help="clouds per GPU per step (default: the BASELINE config's)")
    ap.add_argument("--dist", default="lidar_like", choices=["lidar_like", "uniform"])
    ap.add_argument("--math", default="fp16x3", choices=["fp16x3", "tf32x3"], help="tensor-core arithmetic of the convolutions")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch kernels eagerly instead of replaying a CUDA graph")
    ap.add_argument("--gather-every", type=int, default=0, help="all-gather the detections every G steps (0: once, after the last step)")
    ap.add_argument("--no-nms-c5", action="store_true", help="skip the 100k-box NMS stress (BASELINE configs[4]) leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the detections of the last one as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.wl = WORKLOADS[args.config]
    if args.batch is None:
        args.batch = args.wl["batch"]
    return args


def make_clouds(args, count, seed0, pcr):
    from det3d_b200.utils.synthetic import lidar_like_cloud, uniform_cloud
    fn = lidar_like_cloud if args.dist == "lidar_like" else uniform_cloud
    return [fn(args.wl["n_points"], pcr, args.wl["ndim"], seed0 + i) for i in range(count)]


def build_model(cfg, args):
    """Random-init weights of the named architecture (no checkpoints offline), made to behave like a trained network:
    BatchNorm statistics matched to the activations (features stay O(1)) and heads scaled so that a few % of the
    anchors pass the score threshold -- a realistic top-1000 / NMS workload (utils/synthetic.py)."""
    import torch
    from det3d.models import build_detector
    from det3d_b200.utils.synthetic import calibrate_demo_weights_, demo_weights_
    torch.manual_seed(0)
    model = demo_weights_(build_detector(cfg.model, train_cfg=None, test_cfg=cfg.test_cfg).eval(), 0)
    if torch.cuda.is_available():
        clouds = make_clouds(args, 2, 777, cfg.voxel_generator.range)
        calibrate_demo_weights_(model, cfg, clouds, 0, pass_fraction=args.wl["pass_fraction"])
    return model


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")] + [time.time()])

    def mark(self):
        """Start of the load window: samples read before this moment are dropped."""
        self.t0 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        t0 = getattr(self, "t0", 0.0)
        rows = [r for r in self.rows if r[-1] >= t0] or self.rows[-3:]
        self.rows = rows
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 9 for n, v in zip(names, r[5:9]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU side: the reference's own path on the host cores (SURVEY 8d)
# ---------------------------------------------------------------------------------------------------------------------
def host_cores():
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        pass
    return n


def host_threads(probe=None):
    """Thread count for the CPU leg, whatever torchrun put into OMP_NUM_THREADS (it exports 1 for every rank): all host
    cores are offered, and `probe()` (one forward) picks the count that is actually fastest -- the port is built from many
    small torch / numpy ops, and on a 128-core host 128 threads ran it ~100x SLOWER than 16 (synchronisation overhead)."""
    import torch
    n = host_cores()
    if probe is None:
        torch.set_num_threads(n)
        return n
    best, best_t = n, None
    for c in sorted({c for c in (8, 16, 32, 64, n) if c <= n}):
        torch.set_num_threads(c)
        t0 = time.perf_counter()
        probe()
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def cpu_port(cfg, args, model):
    """CPU restatement of the reference path for this workload (oracle/: spconv and boost are absent from the reference
    checkout, so this leg is a 'port'; its voxelizer stage is the reference's own AOT-compiled kernel when built)."""
    from det3d_b200.core.anchor.anchor_generator import anchors_for_tasks
    from det3d_b200.ops.point_cloud.voxelize import grid_size_of
    grid = grid_size_of(cfg.voxel_generator.voxel_size, cfg.voxel_generator.range)
    anchors = anchors_for_tasks(cfg.target_assigner, grid, cfg.assigner.out_size_factor)
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    if args.config == "second":
        from oracle.second_cpu import SecondCPU as Port
    elif args.config == "pillars":
        from oracle.pillars_cpu import PillarsCPU as Port
    else:
        from oracle.cbgs_cpu import CbgsCPU as Port
    return Port(cfg, sd, anchors)


def _vox_worker(job):
    """One DataLoader-style worker (det3d/datasets/loader/build_loader.py:46-55): voxelizes clouds with the reference
    kernel for `seconds`; returns clouds done."""
    vs, pcr, max_pts, max_vox, n_points, ndim, seed, seconds = job
    from det3d_b200.utils.synthetic import lidar_like_cloud
    from oracle import voxel_ref
    pts = lidar_like_cloud(n_points, pcr, ndim, seed)
    voxel_ref.points_to_voxel(pts, vs, pcr, max_pts, True, max_vox)      # warm (loads the AOT module)
    done, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        voxel_ref.points_to_voxel(pts, vs, pcr, max_pts, True, max_vox)
        done += 1
    return done, time.perf_counter() - t0


def reference_voxelizer_baseline(cfg, args, cores):
    """SURVEY 8d(1): the reference numba voxelizer exactly as VoxelGenerator.generate calls it -- single thread (it is
    single-threaded), full call (incl. the dense lookup map) and loop only, plus one worker process per host core."""
    from oracle import voxel_ref
    if not voxel_ref.available():
        return {"available": False, "why": "oracle/_ref/ref_voxel_aot*.so not built (needs /root/reference at build time)"}
    import multiprocessing as mp
    import numpy as np
    vg = cfg.voxel_generator
    vs, pcr, max_pts, max_vox = list(vg.voxel_size), list(vg.range), vg.max_points_in_voxel, vg.max_voxel_num
    clouds = make_clouds(args, 2, 31, pcr)
    voxel_ref.points_to_voxel(clouds[0], vs, pcr, max_pts, True, max_vox)
    full, n = [], 4
    for i in range(n):
        t0 = time.perf_counter()
        out = voxel_ref.points_to_voxel(clouds[i % 2], vs, pcr, max_pts, True, max_vox)
        full.append(time.perf_counter() - t0)
    bufs = voxel_ref.alloc(vs, pcr, max_pts, max_vox, args.wl["ndim"])
    loop = []
    for i in range(8):
        t0 = time.perf_counter()
        out = voxel_ref.points_to_voxel(clouds[i % 2], vs, pcr, max_pts, True, max_vox, buffers=bufs)
        loop.append(time.perf_counter() - t0)
        voxel_ref.reset(bufs, np.array(out[1]))
    workers = max(1, cores)
    jobs = [(vs, pcr, max_pts, max_vox, args.wl["n_points"], args.wl["ndim"], 100 + w, 3.0) for w in range(workers)]
    try:
        with mp.get_context("spawn").Pool(workers) as pool:
            res = pool.map(_vox_worker, jobs)
        pool_rate = sum(d / t for d, t in res)
    except Exception as e:           # the pool is context, not the product: report and go on
        pool_rate, workers = None, "failed: %s" % e
    return {"available": True, "kind": "reference", "kernel": "det3d/ops/point_cloud/point_cloud_ops.py:7-55 (numba, AOT)",
            "single_thread_full_call_s": statistics.median(full), "single_thread_loop_only_s": statistics.median(loop),
            "single_thread_clouds_per_s": 1.0 / statistics.median(full),
            "pool_workers": workers, "pool_clouds_per_s": pool_rate, "voxels": int(out[1].shape[0])}


def run_reference(args, rank, world):
    """The reference path on the host cores: rank 0 alone, all host threads, the requested warm-up."""
    if rank != 0:
        return
    import torch
    from det3d.torchie import Config
    cfg = Config.fromfile(os.path.join(ROOT, "configs", args.wl["cfg"]))
    model = build_model(cfg, args)
    cpu = cpu_port(cfg, args, model)
    clouds = make_clouds(args, N_CLOUD_POOL, 0, cfg.voxel_generator.range)
    batch = args.batch * world            # the whole job's step, done by the host alone
    cpu.forward([clouds[0]])              # builds the oracle library, warms torch
    cores = host_threads(lambda: cpu.forward([clouds[1]]))
    t0 = time.perf_counter()
    cpu.forward([clouds[0]])
    one = time.perf_counter() - t0
    # a step of the reference arm is a bounded SAMPLE of the job's step: at most `sample` clouds, so that
    # warmup + steps end within a few minutes on any host
    budget = 200.0
    sample = max(1, min(batch, int(budget / max(one, 1e-3) / max(args.steps + args.warmup, 1))))
    for i in range(args.warmup):
        cpu.forward([clouds[(i + j) % N_CLOUD_POOL] for j in range(sample)])
    t0 = time.perf_counter()
    for i in range(args.steps):
        dets = cpu.forward([clouds[(i * sample + j) % N_CLOUD_POOL] for j in range(sample)])
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dets)
    value = args.steps * sample / dt
    line = {
        "impl": "reference", "metric": "point-clouds/sec SECOND SpMiddleFHD @20k pts", "value": value,
        "unit": "clouds/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": "clouds/s", "cores": cores, "kind": "port",
                         "sample": "%d steps x %d cloud(s) of the job's %d-cloud step through the CPU restatement of the "
                                   "reference path (oracle/; spconv and boost are absent from the reference checkout)"
                                   % (args.steps, sample, batch),
                         "host_cores": host_cores(), "stage_seconds": cpu.timings,
                         "reference_voxelizer": reference_voxelizer_baseline(cfg, args, host_cores())},
        "e2e": {"value": value, "unit": "clouds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    _emit(line)


def workload_config(args, world):
    return {"workload": "%s, batch=%d/GPU" % (args.wl["name"], args.batch), "baseline_config": args.config,
            "distribution": args.dist, "points_per_cloud": args.wl["n_points"], "batch_per_gpu": args.batch,
            "global_batch": args.batch * world, "cloud_pool": N_CLOUD_POOL, "l2": "flushed (256 MiB write) between steps",
            "parallelism": "dp%d" % world, "math": "%s tensor-core convolutions (fp32-equivalent)" % args.math,
            "cuda_graph": not args.no_graph,
            "exchange": "one all-gather of the ranks' detections %s, inside the timed region"
                        % ("after the last step" if args.gather_every <= 0 else "every %d steps" % args.gather_every)}


_REAL_STDOUT = None


def _claim_stdout():
    """Route everything libraries write to fd 1 (NCCL prints its version there, build tools chat) to stderr, so that
    stdout carries exactly the one JSON line the contract asks for."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def _emit(line):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (json.dumps(line) + "\n").encode())


DUMP_BUDGET = 64 << 20


def dump_outputs(out_dir, dets):
    """The detections a caller receives for each cloud of one step, as cloud<j>_{box3d_lidar,scores,label_preds}.npy
    (float32; class ids are exact in float32).  Clouds and weights are seeded, so two builds run with the same arguments
    can be compared file for file.  Clouds past DUMP_BUDGET bytes are left out (a fixed prefix of the batch)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for j, det in enumerate(dets):
        arrays = {k: det[k].detach().cpu().numpy().astype(np.float32) for k in ("box3d_lidar", "scores", "label_preds")}
        size = sum(a.nbytes for a in arrays.values())
        if total + size > DUMP_BUDGET:
            print("[bench] --dump-outputs: clouds %d.. left out (%d MiB budget)" % (j, DUMP_BUDGET >> 20), file=sys.stderr)
            break
        total += size
        for k, a in arrays.items():
            np.save(os.path.join(out_dir, "cloud%d_%s.npy" % (j, k)), a)


# ---------------------------------------------------------------------------------------------------------------------
# roofline accounting from the per-stage CUDA events of an eager pass
# ---------------------------------------------------------------------------------------------------------------------
def stage_ms(events, n_steps):
    """(tag -> ms per step, tag -> launches per step, raw list) from _lib.PROFILE_EVENTS."""
    ms, cnt = {}, {}
    for tag, a, b, _info in events:
        ms[tag] = ms.get(tag, 0.0) + a.elapsed_time(b)
        cnt[tag] = cnt.get(tag, 0) + 1
    return {k: v / n_steps for k, v in ms.items()}, {k: v / n_steps for k, v in cnt.items()}


def nms_c5_leg(dev, hbm_peak):
    """BASELINE configs[4]: rotated-BEV NMS of 100k boxes, ours next to the reference's iou3d kernel + host sweep
    (det3d/ops/iou3d/src/iou3d_kernel.cu:250-292 compiled as oracle/_ref, iou3d.cpp:103-116) on the same GPU."""
    import numpy as np
    import torch
    from det3d_b200 import _lib
    from det3d_b200.ops.nms import nms_ops
    from det3d_b200.utils.synthetic import nms_boxes_xyxyr
    n, thr = 100000, 0.2
    boxes, scores = nms_boxes_xyxyr(n, 0, False)
    order = np.argsort(-scores, kind="stable")
    b = torch.from_numpy(boxes[order]).to(dev)
    for _ in range(2):
        keep_idx, keep_count = nms_ops.nms_sorted(b, _lib.BOX_XYXYR, thr)
    torch.cuda.synchronize()
    a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    keep_idx, keep_count = nms_ops.nms_sorted(b, _lib.BOX_XYXYR, thr)
    e.record()
    torch.cuda.synchronize()
    ours_ms = a.elapsed_time(e)
    k = int(keep_count.item())
    pairs = n * (n - 1) / 2
    io_bytes = n * 24 + k * 8
    out = {"boxes": n, "threshold": thr, "kept": k, "ours_ms": ours_ms, "pair_tests_per_s": pairs / (ours_ms * 1e-3),
           "algorithmic_bytes": io_bytes, "mask_bytes_write_plus_read": 2 * n * ((n + 63) // 64) * 8,
           "bound": "fp32 SIMT compute (pair tests), not HBM", "achieved_gbs_io_only": io_bytes / (ours_ms * 1e-3) / 1e9,
           "peak_gbs": hbm_peak}
    try:
        from oracle import iou3d_ref
        if iou3d_ref.available():
            iou3d_ref.nms_mask(b[:4096], thr)                       # warm
            t0 = time.perf_counter()
            mask = iou3d_ref.nms_mask(b, thr)                        # the reference kernel, legacy stream, synchronises
            t1 = time.perf_counter()
            host = mask.cpu().numpy()                                # the reference's 1.25 GB D2H (iou3d.cpp:98-101)
            t2 = time.perf_counter()
            keep_ref = iou3d_ref.host_sweep_c(host)
            t3 = time.perf_counter()
            out["reference"] = {"what": "reference iou3d nms_kernel (compiled from its own source as oracle/_ref) + D2H of the "
                                        "bitmask + host sweep (C restatement of iou3d.cpp:103-116)",
                                "kernel_ms": (t1 - t0) * 1e3, "d2h_ms": (t2 - t1) * 1e3, "host_sweep_ms": (t3 - t2) * 1e3,
                                "total_ms": (t3 - t0) * 1e3, "kept": int(keep_ref.shape[0]),
                                "keep_list_equal": bool(keep_ref.shape[0] == k and np.array_equal(keep_ref, keep_idx[:k].cpu().numpy()))}
            out["speedup_vs_reference_gpu"] = out["reference"]["total_ms"] / ours_ms
    except Exception as ex:     # the comparison leg is context; never fail the bench line on it
        out["reference"] = {"unavailable": "%s: %s" % (type(ex).__name__, ex)}
    return out


def main():
    args = parse()
    _claim_stdout()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from det3d.torchie import Config
    from det3d_b200 import _lib
    from det3d_b200.apis import InferencePipeline, all_gather_detections, init_from_env

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: det3d_b200 has no CPU fallback")
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"      # keep stdout to the single JSON line (NCCL prints its version there)
    rank, world, local = init_from_env()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    cfg = Config.fromfile(os.path.join(ROOT, "configs", args.wl["cfg"]))
    pipe = InferencePipeline(cfg, model=build_model(cfg, args), device=dev)
    pipe.model.set_math(args.math)
    use_graph = not args.no_graph
    B, NP, ND = args.batch, args.wl["n_points"], args.wl["ndim"]
    clouds_np = make_clouds(args, N_CLOUD_POOL, 1000 * rank, cfg.voxel_generator.range)
    pinned = [torch.from_numpy(c).pin_memory() for c in clouds_np]
    resident = [torch.from_numpy(c).to(dev) for c in clouds_np]
    offsets = [NP * i for i in range(B + 1)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    e2e_pts = torch.empty((NP * B, ND), dtype=torch.float32, device=dev)
    dev_pts = torch.empty((NP * B, ND), dtype=torch.float32, device=dev)
    state = {"ring": None, "out_pinned": None, "gathered_pinned": None, "flag_pinned": torch.zeros(1, dtype=torch.int32).pin_memory(),
             "overflowed": False}

    def batch_ids(step):
        return [(step * B + j) % N_CLOUD_POOL for j in range(B)]

    def forward(pts):
        return pipe.forward_graphed(pts, offsets) if use_graph else pipe.pack(pipe.forward_device(pts, offsets))

    def ring_for(packed, steps):
        if state["ring"] is None or state["ring"].shape[0] < steps or state["ring"].shape[1:] != packed.shape:
            state["ring"] = torch.zeros((steps,) + tuple(packed.shape), dtype=torch.float32, device=dev)
        return state["ring"]

    def exchange(n_rows, e2e):
        """The job's one exchange step: all ranks' detections of the last `n_rows` steps, gathered over NCCL."""
        g = all_gather_detections(state["ring"][:n_rows].reshape(n_rows * B, *state["ring"].shape[2:]))
        if e2e:
            if state["gathered_pinned"] is None or state["gathered_pinned"].numel() < g.numel():
                state["gathered_pinned"] = torch.empty(g.numel(), dtype=torch.float32, pin_memory=True)
            state["gathered_pinned"][:g.numel()].view(g.shape).copy_(g, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        return g

    def step_device(step, steps):
        ids = batch_ids(step)
        if B == 1:
            pts = resident[ids[0]]
        else:
            for j, i in enumerate(ids):
                dev_pts[j * NP:(j + 1) * NP].copy_(resident[i], non_blocking=True)
            pts = dev_pts
        packed = forward(pts)
        ring_for(packed, steps)[step % steps].copy_(packed, non_blocking=True)

    def step_e2e(step, steps):
        ids = batch_ids(step)
        for j, i in enumerate(ids):
            e2e_pts[j * NP:(j + 1) * NP].copy_(pinned[i], non_blocking=True)       # H2D from pinned memory
        packed = forward(e2e_pts)
        ring_for(packed, steps)[step % steps].copy_(packed, non_blocking=True)
        if state["out_pinned"] is None:
            state["out_pinned"] = torch.empty(packed.shape, dtype=torch.float32, pin_memory=True)
        state["out_pinned"].copy_(packed, non_blocking=True)                       # this step's detections to the host
        flag = pipe.overflow_flag()
        if flag is not None:
            state["flag_pinned"].copy_(flag, non_blocking=True)                    # f16-range guard of the FP16x3 kernels
        torch.cuda.current_stream().synchronize()     # the caller holds the detections on the host
        if int(state["flag_pinned"][0]):
            state["overflowed"] = True

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, e2e):
        evs = []
        ge = max(0, args.gather_every)
        barrier()
        for s in range(steps):
            flush.zero_()                                   # L2 flush, outside the timed events
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn(s, steps)
            last = s == steps - 1
            if (ge > 0 and (s + 1) % ge == 0) or (last and (ge <= 0 or steps % ge)):
                exchange(steps if ge <= 0 else ((s % ge) + 1), e2e)
            b.record()
            evs.append((a, b))
        barrier()
        ms = sum(a.elapsed_time(b) for a, b in evs)
        if os.environ.get("D3B_BENCH_DEBUG"):
            print(f"[bench] rank {rank} {'e2e' if e2e else 'device'} per-step ms: "
                  + " ".join(f"{a.elapsed_time(b):.3f}" for a, b in evs), file=sys.stderr)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    warm = max(args.warmup, 3)
    ring_steps = max(warm, args.steps)
    for s in range(warm):
        step_device(s, ring_steps)
        step_e2e(s, ring_steps)
    ge0 = max(0, args.gather_every)
    exchange(args.steps if ge0 <= 0 else min(ge0, args.steps), True)   # same shapes as the timed exchange: the device ring,
    #                                                                  the NCCL buffers and the pinned landing buffer exist
    #                                                                  before the clock starts (cudaHostAlloc alone is ~90 ms)
    if state["overflowed"]:
        raise SystemExit("bench.py: the FP16x3 kernels flagged an f16-range overflow on the synthetic workload; run with --math tf32x3")

    sampler.mark()                      # clocks are sampled from here to the end of the per-kernel pass (same load)
    ms = timed(step_device, args.steps, False)
    ms_e2e = timed(step_e2e, args.steps, True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, pipe.unpack(state["out_pinned"]))       # the last step_e2e, already on the host

    # ---- per-stage pass: eager launches of the SAME kernels, CUDA events around every det3d_b200 call on the
    #      launching stream (voxelize / rulebook / sparse convs / dense convs / predict): launch count + rooflines ----
    n_prof = min(args.steps, 10)

    def step_eager(step, steps):
        ids = batch_ids(step)
        pts = resident[ids[0]] if B == 1 else torch.cat([resident[i] for i in ids])
        packed = pipe.pack(pipe.forward_device(pts, offsets))
        ring_for(packed, steps)[step % steps].copy_(packed, non_blocking=True)

    for s in range(2):
        step_eager(s, n_prof)
    launches0 = _lib.launch_count()
    events = []
    _lib.PROFILE_EVENTS = events
    try:
        timed(step_eager, n_prof, False)
    finally:
        _lib.PROFILE_EVENTS = None
    launches_per_step = (_lib.launch_count() - launches0) / n_prof
    torch.cuda.synchronize()

    # ---- in-graph stage pass: a second capture of the same forward with an external timing event (one event-record node)
    #      at every stage boundary of the main stream; replayed like the timed steps (L2 flushed before each).  These are the
    #      durations the stages have INSIDE the product graph -- the eager pass above adds the host-side cost of every call
    #      (ctypes, two tensor-map encodes per dense layer, launch latency) between its events. ----
    graph_ms = {}
    if use_graph and world == 1:       # (N > 1: a second capture next to a live NCCL communicator is not worth the risk;
        #                                 the N = 1 line carries the rooflines)
        pipe._graphs.clear()
        _lib.GRAPH_MARKS = marks = []
        try:
            n_rep = n_prof + 2
            for s in range(n_rep):
                ids = batch_ids(s)
                pts = resident[ids[0]] if B == 1 else torch.cat([resident[i] for i in ids])
                flush.zero_()
                pipe.forward_graphed(pts, offsets)
                torch.cuda.synchronize()
                if s >= 2:
                    for (tag, ev, _st), (_t1, ev1, _s1) in zip(marks[:-1], marks[1:]):
                        graph_ms[tag] = graph_ms.get(tag, 0.0) + ev.elapsed_time(ev1) / (n_rep - 2)
        except RuntimeError as ex:        # (timing of externally recorded events unsupported: keep the eager numbers)
            print("[bench] in-graph stage pass unavailable: %s" % ex, file=sys.stderr)
            graph_ms = {}
        finally:
            _lib.GRAPH_MARKS = None
            pipe._graphs.clear()
    clocks = sampler.stop() if rank == 0 else None

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    bf16_peak = float(peaks.get("bf16_tflops", 1590.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    traffic = {}
    try:      # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` captures
        traffic = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
    except OSError:
        pass
    traffic_note = "static: from the committed ncu --set full capture (profiles/r2_traffic.json), not measured by this run"
    ms_step = ms / args.steps
    st_ms, st_cnt = stage_ms(events, n_prof)
    timing = "CUDA events around each call on its launching stream, eager pass of %d steps" % n_prof
    rooflines = {}

    # --- dense BEV convolutions (tensor bound) ---
    bev = [(tag, a.elapsed_time(b), info) for tag, a, b, info in events if tag in ("bev3x3", "bev1x1", "deblock", "heads")]
    dom = [x for x in bev if x[0] == "bev3x3" and x[2].get("flops")]
    if dom:
        # the most expensive 3x3 shape of the step is the dominant kernel
        by_shape = {}
        for _tag, t, info in dom:
            key = (info["c_in"], info["c_out"], info["stride"], info["pixels_out"])
            d = by_shape.setdefault(key, {"ms": 0.0, "n": 0, "info": info})
            d["ms"] += t
            d["n"] += 1
        key, d = max(by_shape.items(), key=lambda kv: kv[1]["ms"])
        launch_ms = d["ms"] / d["n"]
        launch_ms_eager = launch_ms
        if graph_ms.get("bev3x3"):
            # inside the graph: the 3x3 group's duration, split over its shapes in the proportion of the eager pass
            launch_ms = graph_ms["bev3x3"] * (d["ms"] / sum(x[1] for x in dom)) / (d["n"] / n_prof)
            timing = ("external CUDA timing events (event-record graph nodes) at the boundaries of the 3x3 group inside the "
                      "replayed CUDA graph, %d replays, L2 flushed before each; eager-pass time per launch (host cost of the "
                      "call between the events): %.4f ms" % (n_prof, launch_ms_eager))
        flops = d["info"]["flops"]
        tensor_peak, tensor_peak_kind = bf16_peak, "burst (kernel timed alone)"
        if graph_ms.get("bev3x3") and peaks.get("bf16_tflops_sustained"):
            # timed inside the replayed step: the sustained cuBLAS figure is the denominator (MEASURED_PEAKS.json: burst for a
            # kernel timed alone, sustained for a kernel timed inside a long step)
            tensor_peak, tensor_peak_kind = float(peaks["bf16_tflops_sustained"]), "sustained (kernel timed inside the replayed step)"
        tf = flops / (launch_ms * 1e-3) / 1e12
        per_math = 3.0 if args.math == "fp16x3" else 6.0       # bf16-peak-equivalents spent per fp32-equivalent flop
        rooflines["roofline"] = {
            "kernel": ("d3b::bev_conv16_cs_kernel (channel-stationary M128 x N256 tiles): dense BEV conv3x3 %d->%d (RPN), %d launches/step"
                       % (key[0], key[1], d["n"] // n_prof)
                       if ((_lib.lib().d3b_get_bev_variant() == 1 or (_lib.lib().d3b_get_bev_variant() == 2 and d["info"].get("tiles", 0) >= 296))
                           and key[2] == 1 and key[1] % 128 == 0 and key[0] % 64 == 0) else
                       "d3b::bev_conv16_kernel<3,%d,%d>: dense BEV conv3x3 %d->%d (RPN), %d launches/step"
                       % (key[2], min(key[1], 128), key[0], key[1], d["n"] // n_prof)) if args.math == "fp16x3" else
                      "d3b::spconv_tc_kernel<128>: dense BEV conv3x3 (RPN, tf32x3 path), %d launches/step" % (d["n"] // n_prof),
            "bound": "tensor", "achieved": tf, "peak": tensor_peak, "unit": "TFLOP/s", "frac": tf / tensor_peak,
            "peak_kind": tensor_peak_kind, "frac_of_burst_peak": tf / bf16_peak,
            "traffic": traffic.get("bev3x3_dram_bytes_per_launch"), "traffic_note": traffic_note, "peak_source": peak_src,
            "algorithmic_flops_per_launch": flops,
            "algorithmic_bytes_per_launch": d["info"]["pixels_in"] * key[0] * 4 + key[3] * key[1] * 4 + 9 * key[0] * key[1] * 4,
            "launch_ms": launch_ms, "launches_per_step": d["n"] // n_prof,
            "share_of_step": launch_ms * (d["n"] / n_prof) / ms_step, "timing": timing,
            "note": "fp32-equivalent flops (the reference runs this layer as fp32 cuDNN).  %s reaches fp32 accuracy with 3 "
                    "split products per flop on the %s pipe, so the ceiling of the algorithm is peak/%d and tensor-pipe "
                    "utilisation is %d x frac = %.2f" % (args.math, "f16" if args.math == "fp16x3" else "tf32 (half rate)",
                                                         int(per_math), int(per_math), per_math * tf / tensor_peak),
            "bev_stack": {"launches_per_step": len(bev) // n_prof, "flops_per_step": sum(x[2].get("flops", 0) for x in bev) // n_prof,
                          "kernel_ms_per_step": sum(x[1] for x in bev) / n_prof,
                          "share_of_step": sum(x[1] for x in bev) / n_prof / ms_step}}

    timing = "CUDA events around each call on its launching stream, eager pass of %d steps" % n_prof
    # --- sparse middle encoder (HBM / latency bound) ---
    fused = getattr(pipe.model.backbone, "fused", None)
    if fused is not None and "sparse" in st_ms:
        enc = fused().accounting()
        enc_ms = st_ms["sparse"]
        enc_timing = timing
        if graph_ms.get("sparse"):
            enc_ms = graph_ms["sparse"]
            enc_timing = ("external CUDA timing events inside the replayed graph: first sparse convolution .. first dense layer "
                          "(the 14 launches, the waits on the rulebook side stream and the scatter into the BEV planes); "
                          "eager-pass sum of the 14 calls: %.4f ms" % st_ms["sparse"])
        gbs = enc["bytes"] / (enc_ms * 1e-3) / 1e9
        rooflines["roofline_encoder"] = {
            "kernel": ("d3b::spconv_os16_kernel (output-stationary FP16x3, deterministic)" if args.math == "fp16x3" else
                       "d3b::spconv_pairs_kernel (tf32x3, fp32 atomics)") + ": sparse middle encoder, %d launches/step" % len(enc["layers"]),
            "bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
            "traffic": traffic.get("encoder_dram_bytes_per_step"), "traffic_note": traffic_note, "peak_source": peak_src,
            "algorithmic_bytes_per_step": enc["bytes"], "flops_per_step": enc["flops"], "kernel_ms_per_step": enc_ms,
            "share_of_step": enc_ms / ms_step, "timing": enc_timing,
            "note": "below the tensor ridge by construction (2..32 flop/B, SURVEY 8d); at ~100-160 output tiles per layer the "
                    "bound is the 27-offset dependent chain per tile (gather latency), not DRAM"}
        # --- rulebook (HBM / latency bound) ---
        if "rulebook" in st_ms:
            rb_bytes, seen = 0, set()
            for lvl, rb, _L in fused().last_levels():
                if id(rb) in seen:
                    continue
                seen.add(id(rb))
                n_in, n_out = int(rb.in_level.n[0].item()), int(rb.out_level.n[0].item())
                pairs = int((rb.nbr[:, :n_out] >= 0).sum().item()) if n_out else 0
                rb_bytes += n_in * 16 + pairs * 8 + n_out * 16           # SURVEY 8d: coords in + pairs out + coords out
            gbs = rb_bytes / (st_ms["rulebook"] * 1e-3) / 1e9
            rooflines["roofline_rulebook"] = {
                "kernel": "d3b rulebook chain (hash insert, neighbour map, bitmap mark / scan / emit), %d calls/step on a side stream"
                          % int(st_cnt["rulebook"]),
                "bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak, "traffic": None,
                "algorithmic_bytes_per_step": rb_bytes, "kernel_ms_per_step": st_ms["rulebook"], "timing": timing,
                "note": "latency bound: a few hundred KB per call; overlapped with the convolutions (side stream) in the product path"}

    # --- voxelizer (HBM / latency bound) ---
    if "voxelize" in st_ms:
        counts = pipe.voxelizer._bufs[next(iter(pipe.voxelizer._bufs))]["counts"]
        m = int(counts[B].item())
        vg = cfg.voxel_generator
        full_bytes = B * NP * ND * 4 + m * (vg.max_points_in_voxel * ND * 4 + 12 + 4)         # SURVEY 8d B_vox
        fused_bytes = B * NP * ND * 4 + m * (ND * 4 + 12 + 4)                                 # mean fused, voxels not materialised
        alg = full_bytes if pipe._reader_takes_points else fused_bytes
        gbs = alg / (st_ms["voxelize"] * 1e-3) / 1e9
        rooflines["roofline_voxelize"] = {
            "kernel": "d3b voxelizer (vox_insert / chunk count-scan-assign / vox_lists / vox_emit), one d3b_voxelize call/step",
            "bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak, "traffic": None,
            "algorithmic_bytes_per_step": alg, "algorithmic_bytes_reference_outputs": full_bytes, "voxels": m,
            "kernel_ms_per_step": st_ms["voxelize"], "share_of_step": st_ms["voxelize"] / ms_step, "timing": timing,
            "note": "latency bound: ~1-2 MB per cloud across six dependent launches; bytes follow SURVEY 8d (inputs read once + "
                    "outputs written once; the per-voxel point lists are not materialised when the reader only needs the mean)"}

    # --- predict + NMS at the detector's operating point ---
    if "predict" in st_ms:
        pre = max(info.get("pre", 0) for tag, _a, _b, info in events if tag == "predict")
        tasks = int(round(st_cnt["predict"]))
        pairs = B * tasks * pre * (pre - 1) / 2
        rooflines["roofline_nms"] = {
            "kernel": "d3b_predict_task (head scores -> top-k -> decode -> rotated NMS mask + sweep -> finalize), %d call(s)/step" % tasks,
            "bound": "fp32 SIMT compute / latency", "kernel_ms_per_step": st_ms["predict"], "share_of_step": st_ms["predict"] / ms_step,
            "candidates": pre, "pair_tests_per_s_upper": pairs / (st_ms["predict"] * 1e-3), "timing": timing}

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    clouds_per_step = B * world
    value = clouds_per_step * args.steps / (ms * 1e-3)
    e2e_value = clouds_per_step * args.steps / (ms_e2e * 1e-3)
    d2h = int(state["out_pinned"].numel() * 4) + 4 + int(state["gathered_pinned"].numel() * 4 / args.steps)
    line = {
        "metric": "point-clouds/sec SECOND SpMiddleFHD @20k pts" if args.config == "second" else "point-clouds/sec " + args.wl["name"],
        "value": value, "unit": "clouds/s",
        "n_gpus": world, "steps": args.steps, "warmup": warm, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world),
        "e2e": {"value": e2e_value, "unit": "clouds/s", "h2d_bytes_per_step": B * NP * ND * 4,
                "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(round(launches_per_step * args.steps)), "gpu_launches_per_step": launches_per_step,
        "gpu_launches_note": ("det3d_b200 kernels per step counted by d3b_launch_count() in an eager pass; the timed region replays "
                              "the same kernel nodes from a CUDA graph") if use_graph else "counted in an eager pass",
        "clocks": clocks, "stage_ms_per_step": st_ms, "stage_calls_per_step": st_cnt,
        "stage_ms_per_step_in_graph": graph_ms or None,
    }
    line.update(rooflines)
    if "roofline" not in line and "roofline_encoder" in line:
        line["roofline"] = line["roofline_encoder"]
    if world == 1 and not args.no_nms_c5:
        line["nms_c5"] = nms_c5_leg(dev, hbm_peak)
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_port(cfg, args, pipe.model)
        cpu.forward([clouds_np[0]])
        cores = host_threads(lambda: cpu.forward([clouds_np[1]]))
        n_cpu = 3
        t0 = time.perf_counter()
        for i in range(n_cpu):
            cpu.forward([clouds_np[i % N_CLOUD_POOL]])
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": n_cpu / dt, "unit": "clouds/s", "cores": cores, "kind": "port",
                                "sample": "%d full forwards of one %d-point cloud through the CPU restatement of the reference "
                                          "path (oracle/); voxelizer stage also timed on the reference's own kernel" % (n_cpu, NP),
                                "host_cores": host_cores(), "stage_seconds": cpu.timings,
                                "reference_voxelizer": reference_voxelizer_baseline(cfg, args, host_cores())}
    _emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
