#!/usr/bin/env python
"""Benchmark of the MVSNeRF render hot path (BASELINE.json metric: rays/s @ 128 samples, DTU 512x640).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--mode fp32] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic rays: one full 512x640 frame
(327 680 rays x 128 samples) per GPU rendered against a resident encoding volume -- the
reference's own frame loop (renderer_video.ipynb "DTU video rendering": the volume is built once per
scene, frames are then rendered from it).  Every step renders a different target camera of a
seeded spiral path.  The once-per-scene volume build (FeatureNet + cost volume + CostRegNet) is
timed separately and reported under "volume_build".

value      : whole-job rays/s with the rays already resident in HBM (kernel launch only).
e2e        : the same metric through the host-buffer call (pinned host rays -> H2D -> kernel ->
             D2H of rgb+depth), copies inside the timed region.
roofline   : the render kernel's algorithmic FLOPs (32 178 176 per ray, SURVEY.md 8(d)) over its
             CUDA-event duration, against the measured bf16 tensor peak (MEASURED_PEAKS.json).
cpu_baseline / --impl reference : the CPU restatement of the reference path (oracle/, PyTorch CPU,
             all host threads) on a bounded sample of the same workload.

--dump-outputs DIR : after the timed steps, the frame the last one rendered (single GPU): DIR/rgb.npy [H*W, 3] and
             DIR/depth.npy [H*W], float32.  The scene, weights and cameras are seeded, so two builds run with the
             same arguments can be compared output for output.

Multi-GPU (torchrun, one rank per GPU): rays shard across ranks, the volume is replicated, one
NCCL all-gather of rgb+depth per step sits inside the timed region; weak scaling (one frame per
GPU per step).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

H, W, PAD, S = 512, 640, 24, 128
N_RAYS = H * W
FLOP_PER_RAY = 32_178_176          # 128 x 251 392 MLP FLOPs           (SURVEY.md 8(d), BASELINE.md 2)
BYTES_PER_RAY = 51_248             # 128 x 400 B gather + 32 B in + 16 B out
SPLIT_EXEC = 109_312 / 125_696     # MACs per sample the split kernel executes after folding feature_linear into the views layer
WEIGHTS = os.path.join(ROOT, "tests", "golden", "mvsnerf_v0_weights.npz")
METRIC = "rays/sec @ 128 samples, DTU 512x640"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"],
                    bf16_tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region.

    nvidia-smi needs a few hundred ms to come up, longer than a short timed region, so the process is started early
    (before the scene is built) and streams one line every 25 ms; every line is stamped on arrival and only the lines
    that arrived inside the marked window [begin(), end()] are used."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines, self.thread = index, None, [], None
        self.t0 = self.t1 = None

    def start(self):
        import threading
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "25", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, bufsize=1)
        except OSError:
            self.proc = None
            return

        def pump():
            for line in self.proc.stdout:
                self.lines.append((time.perf_counter(), line))
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def begin(self):
        self.t0 = time.perf_counter()

    def end(self):
        self.t1 = time.perf_counter()

    def in_window(self):
        t1 = self.t1 if self.t1 is not None else time.perf_counter()
        return sum(1 for t, _ in list(self.lines) if self.t0 is not None and self.t0 <= t <= t1)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        if self.thread is not None:
            self.thread.join(timeout=2)
        t0 = self.t0 if self.t0 is not None else 0.0
        t1 = self.t1 if self.t1 is not None else float("inf")
        sm, mx, reasons = [], [], set()
        for t, line in list(self.lines):
            if not (t0 <= t <= t1):
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"], "lines_total": len(self.lines)}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------
# CPU reference arm (the oracle port on the host cores)
# ---------------------------------------------------------------------------------------------
def cpu_reference_setup():
    from oracle import mvsnerf_oracle as orc
    from mvsnerf_b200 import synthetic
    torch.set_num_threads(min(32, os.cpu_count() or 1))   # big hosts: the intra-op pool regresses past ~32 threads
    weights = orc.load_weights_npz(WEIGHTS)
    sc = synthetic.make_scene(H, W, pad=PAD, seed=0)
    return orc, synthetic, weights, sc


def cpu_pick_threads(orc, weights, sc, rays, volume):
    """Give the CPU arm its best configuration: PyTorch's intra-op pool stops scaling (and then
    regresses) well below the core count of a big host, so try a few pool sizes on a small sample
    and keep the fastest.  Returns the thread count used from here on."""
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu})
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        cpu_render_sample(orc, weights, sc, rays[:256], volume)
        t = cpu_render_sample(orc, weights, sc, rays[:1024], volume)
        if t < best_t:
            best, best_t = c, t
    torch.set_num_threads(best)
    return best


def cpu_render_sample(orc, weights, sc, rays, volume):
    t0 = time.perf_counter()
    with torch.no_grad():
        orc.render_rays(rays, volume, sc.imgs_raw, sc.pose_source, weights, H, W, sc.near_far, float(PAD),
                        n_samples=S, chunk=5120)
    return time.perf_counter() - t0


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port: the reference
    is pure Python/PyTorch and /root/reference does not exist on the GPU box), all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    orc, synthetic, weights, sc = cpu_reference_setup()
    cores = os.cpu_count() or 1
    sample = 2048
    with torch.no_grad():
        t0 = time.perf_counter()
        volume = orc.encode_volume(sc.imgs_norm, sc.proj_mats, sc.near_far, PAD, weights)
        t_vol = time.perf_counter() - t0
    path = synthetic.spiral_path(sc, max(args.steps + args.warmup, 2))
    threads = cpu_pick_threads(orc, weights, sc, synthetic.scene_rays(sc)[::37][:2048].contiguous(), volume)
    times = []
    for i in range(args.warmup + args.steps):
        rays = synthetic.scene_rays(sc, path[i % len(path)])
        g = torch.Generator().manual_seed(i)
        rays = rays[torch.randperm(N_RAYS, generator=g)[:sample]].contiguous()
        dt = cpu_render_sample(orc, weights, sc, rays, volume)
        if i >= args.warmup:
            times.append(dt)
    t = sum(times) / len(times)
    value = sample / t
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": {"workload": "DTU-shaped 512x640 frame, 3 source views, pad 24, N_samples=128, volume resident",
                   "sample": f"{sample} random rays of the frame per step (bounded sample; rays/s is per-ray linear)"},
        "cpu_baseline": {"value": value, "unit": "rays/s", "cores": threads, "host_cpus": cores, "kind": "port",
                         "sample": f"{sample} rays x 128 samples per step, chunk 5120, torch {torch.__version__} CPU, "
                                   f"{torch.get_num_threads()} threads; volume build once: {t_vol:.1f} s"},
        "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "volume_build": {"ms": t_vol * 1e3},
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
MODE_DTYPE = {"fp32": "fp32", "half": "fp16 operands / fp32 accumulate", "pair": "fp16 operands / fp32 accumulate",
              "split": "2x fp16 split operands / fp32 accumulate"}
MODE_KERNEL = {"fp32": "render_fp32_kernel", "half": "render_tc_kernel", "pair": "render_tc2_kernel",
               "split": "render_tcs_kernel"}


def _median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2] if xs else None


def run_ours(args):
    import torch.distributed as dist
    from mvsnerf_b200 import backend, synthetic, lib
    from mvsnerf_b200 import distributed as mdist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback; "
                         "use --impl reference for the CPU arm)")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    modes = {"fp32": lib.MLP_FP32, "half": lib.MLP_TC_HALF, "split": lib.MLP_TC_SPLIT, "pair": lib.MLP_TC_PAIR}
    mode = modes[args.mode]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                 # early: nvidia-smi is streaming by the time the timed region begins

    fn, mvs = backend.MVSNeRF().to(dev), backend.MVSNet().to(dev).train()
    backend.load_weights_npz(fn, mvs, WEIGHTS)
    sc = synthetic.make_scene(H, W, pad=PAD, seed=0)
    d = sc.to(dev)
    main = torch.cuda.current_stream()

    def ev():
        return torch.cuda.Event(enable_timing=True)

    def ev_time(f, reps):
        ts = []
        for _ in range(reps):
            a, b = ev(), ev()
            a.record(); f(); b.record(); b.synchronize()
            ts.append(a.elapsed_time(b))
        return ts

    def max_over_ranks(x):
        t = torch.tensor([float(x)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- once-per-scene encoding volume (reported, not part of the step) -----------------------
    with torch.no_grad():
        vol, _, _ = mvs(d.imgs_norm, d.proj_mats, sc.near_far, pad=PAD)            # warm-up + result
        torch.cuda.synchronize()
        t_build = min(ev_time(lambda: mvs(d.imgs_norm, d.proj_mats, sc.near_far, pad=PAD), 3))
        t_feat = min(ev_time(lambda: mvs.feature(d.imgs_norm.reshape(3, 3, H, W)), 3))
        feats = mvs.feature(d.imgs_norm.reshape(3, 3, H, W)).view(1, 3, 32, H // 4, W // 4)
        dv = torch.linspace(sc.near_far[0], sc.near_far[1], 128, device=dev)[None]
        t_cost = min(ev_time(lambda: mvs.build_volume_costvar_img(d.imgs_norm, feats, d.proj_mats, dv, pad=PAD), 3))
        cost, _ = mvs.build_volume_costvar_img(d.imgs_norm, feats, d.proj_mats, dv, pad=PAD)
        t_reg = min(ev_time(lambda: mvs.cost_reg_2(cost), 3))
        del cost, feats
    pk = peaks()
    nvox = 128 * (H // 4 + 2 * PAD) * (W // 4 + 2 * PAD)

    def render(rays, m=mode, out=None, sink=None, n_samples=S):
        return backend.render_rays(rays, vol, d.imgs_raw, d.pose_source, fn, sc.near_far, float(PAD),
                                   N_samples=n_samples, mlp_mode=m, out=out, sink=sink)

    # ---- frame assembly across ranks: NVLink peer stores from the kernel epilogue, else ONE NCCL all-gather ----
    assemble, frame, why = "none", None, None
    if world > 1:
        assemble = args.assemble
        if assemble == "peer":
            ok = 1.0
            try:
                frame = mdist.PeerFrame(world * N_RAYS, n_buffers=2)
            except Exception as e:                                   # no peer access on this box: say so, use NCCL
                ok, why = 0.0, f"{type(e).__name__}: {e}"
            t = torch.tensor([ok], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            if float(t.item()) < 1.0:
                frame, assemble = None, "nccl"
                why = why or "a peer rank could not map the frame buffers"

    # ---- frames: a spiral of target cameras, each rank renders its own frame of every step ------
    n_frames = args.warmup + args.steps
    n_distinct = min(n_frames, 16)                     # distinct target cameras kept resident (cycled for long runs)
    path = synthetic.spiral_path(sc, max(n_distinct * world, 2))
    rays_host = [synthetic.scene_rays(sc, path[(i * world + rank) % len(path)]).pin_memory() for i in range(n_distinct)]
    rays_dev = [r.to(dev) for r in rays_host]
    rgb = torch.empty(N_RAYS, 3, device=dev)
    depth = torch.empty(N_RAYS, device=dev)
    px_local = torch.empty(N_RAYS, 4, device=dev)
    px_all = torch.empty(world * N_RAYS, 4, device=dev) if assemble == "nccl" else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)                  # > 126 MB L2
    launches = [0]
    local_sink = lib.PeerSink()                                                    # NCCL path: one [n,4] send buffer
    local_sink.frame[0], local_sink.n_peers, local_sink.first_pixel = px_local.data_ptr(), 1, 0

    def step(i, m=mode, kev=None):
        """One step: this rank's frame through the render kernel; at N > 1 the job's frames assembled on every rank."""
        r = rays_dev[i % n_distinct]
        if kev:
            kev[0].record()
        if assemble == "peer":
            render(r, m, sink=frame.sink(rank * N_RAYS))
        elif assemble == "nccl":
            render(r, m, sink=local_sink)                # packed (r,g,b,depth) texels straight from the epilogue
        else:
            render(r, m, out=(rgb, depth))
        if kev:
            kev[1].record()
        launches[0] += 1
        if assemble == "peer":
            frame.complete()
            frame.rotate()
        elif assemble == "nccl":
            dist.all_gather_into_tensor(px_all, px_local)

    def timed_steps(m, n_warm, n_steps):
        """-> (ms_per_step max over ranks, kernel ms list of THIS rank on the same launches, per-step (kernel, rest) ms)."""
        for i in range(n_warm):
            step(i, m)
        barrier()
        evs = []
        for i in range(n_warm, n_warm + n_steps):
            flush.zero_()                                                          # L2 flush, untimed
            a, ka, kb, b = ev(), ev(), ev(), ev()
            a.record(); step(i, m, (ka, kb)); b.record()
            evs.append((a, ka, kb, b))
        barrier()
        tot = sum(a.elapsed_time(b) for a, _, _, b in evs)
        kern = [ka.elapsed_time(kb) for _, ka, kb, _ in evs]
        rest = [kb.elapsed_time(b) for _, _, kb, b in evs]
        return max_over_ranks(tot) / n_steps, kern, rest

    with torch.no_grad():
        for i in range(args.warmup):
            step(i)
        barrier()
        launches[0] = 0
        sampler.begin()
        t_wall0 = time.perf_counter()
        ms_per_step, kern_list, rest_list = timed_steps(mode, 0, args.steps)
        t_wall = time.perf_counter() - t_wall0
        n_launch = launches[0]
        # the caller's view of the last timed step; the steps below render into the same buffers
        last_frame = (rgb.clone(), depth.clone()) if args.dump_outputs else None
        # a timed region shorter than a few sampling periods may have caught no clock sample: keep the SAME load running
        # (untimed, same number of extra steps on every rank) until the window is at least 0.4 s long
        t_region = ms_per_step * 1e-3 * args.steps                 # max over ranks: identical on every rank
        if t_region < 0.4:
            for i in range(int(math.ceil((0.4 - t_region) / (ms_per_step * 1e-3)))):
                step(i, mode)
            barrier()
        sampler.end()
        clocks = sampler.stop() if rank == 0 else None
        if clocks is not None and t_region < 0.4:
            clocks["window"] = "timed region + the same steps continued untimed to 0.4 s"
        value = world * N_RAYS / (ms_per_step * 1e-3)
        kern = sum(kern_list) / len(kern_list)        # the render kernel alone, on the SAME launches as ms_per_step

        # per-rank trace of the step's two parts (what a scaling loss would have to come from)
        trace = None
        if world > 1:
            mine = torch.tensor([_median(kern_list), max(kern_list), _median(rest_list), max(rest_list)], device=dev,
                                dtype=torch.float64)
            allr = torch.empty(world, 4, device=dev, dtype=torch.float64)
            dist.all_gather_into_tensor(allr, mine)
            trace = {"render_ms_median_per_rank": [round(float(x), 4) for x in allr[:, 0]],
                     "render_ms_max_per_rank": [round(float(x), 4) for x in allr[:, 1]],
                     "assembly_ms_median_per_rank": [round(float(x), 4) for x in allr[:, 2]],
                     "assembly_ms_max_per_rank": [round(float(x), 4) for x in allr[:, 3]],
                     "note": "CUDA events per step on each rank: render = the kernel launch (with its peer stores), "
                             "assembly = what follows it inside the step (peer: 1-element barrier; nccl: pack + all-gather), "
                             "including the wait for the slowest rank"}

        # ---- the NCCL alternative on the same steps, for the record (peer-store runs only) ----------------------
        alt = None
        if assemble == "peer" and not args.no_assembly_comparison:
            assemble = "nccl"
            px_all = torch.empty(world * N_RAYS, 4, device=dev)
            ms_n, kern_n, rest_n = timed_steps(mode, 3, args.steps)
            alt = {"assemble": "one NCCL all_gather_into_tensor of packed [n,4] pixels per step", "ms_per_step": ms_n,
                   "value": world * N_RAYS / (ms_n * 1e-3), "unit": "rays/s",
                   "render_ms_median": _median(kern_n), "assembly_ms_median": _median(rest_n), "assembly_ms_max": max(rest_n)}
            assemble = "peer"
            px_all = None

        # ---- e2e: host rays -> H2D -> kernel -> (assembly) -> D2H, through the host-buffer call ---------
        def e2e_run(m, n_steps):
            hfr = backend.HostFrameRenderer(N_RAYS, dev)

            def one(i):
                if assemble == "peer":
                    hfr.render(rays_host[i % n_distinct], vol, d.imgs_raw, d.pose_source, fn, sc.near_far, float(PAD),
                               N_samples=S, mlp_mode=m, sink=frame.sink(rank * N_RAYS), after_launch=frame.complete)
                    frame.rotate()
                elif assemble == "nccl":
                    hfr.render(rays_host[i % n_distinct], vol, d.imgs_raw, d.pose_source, fn, sc.near_far, float(PAD),
                               N_samples=S, mlp_mode=m, sink=local_sink,
                               after_launch=lambda: dist.all_gather_into_tensor(px_all, px_local))
                else:
                    hfr.render(rays_host[i % n_distinct], vol, d.imgs_raw, d.pose_source, fn, sc.near_far, float(PAD),
                               N_samples=S, mlp_mode=m)
            for i in range(2):
                one(i)
            barrier()
            t0 = time.perf_counter()
            for i in range(n_steps):
                one(args.warmup + i)
            barrier()
            t = max_over_ranks(time.perf_counter() - t0)
            return world * N_RAYS * n_steps / t, hfr
        e2e_value, hfr = e2e_run(mode, args.steps)

        # the same loop fed the way the reference's video notebook feeds it: one camera pose per frame from the host, rays
        # generated on the device (data/ray_utils.get_rays -> mvsn_make_rays); reported beside `e2e`, not instead of it
        e2e_cam = None
        if world == 1:
            poses = [path[(args.warmup + i) % len(path)].pin_memory() for i in range(args.steps)]
            for i in range(2):
                hfr.render_camera(poses[i % len(poses)], d.directions, vol, d.imgs_raw, d.pose_source, fn, sc.near_far, float(PAD),
                                  N_samples=S, mlp_mode=mode)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(args.steps):
                hfr.render_camera(poses[i], d.directions, vol, d.imgs_raw, d.pose_source, fn, sc.near_far, float(PAD),
                                  N_samples=S, mlp_mode=mode)
            torch.cuda.synchronize()
            e2e_cam = {"value": N_RAYS * args.steps / (time.perf_counter() - t0), "unit": "rays/s", "h2d_bytes_per_step": 64,
                       "d2h_bytes_per_step": hfr.d2h_bytes,
                       "api": "HostFrameRenderer.render_camera: pinned c2w -> H2D -> mvsn_make_rays -> mvsn_render_rays -> D2H"}

        # ---- strong scaling (BASELINE configs 2 and 4 as ONE job): one frame / one 4096-ray batch sharded over the
        # ranks through the shipped API (distributed.render_rays_sharded), bit-equal to the single-GPU result ----
        strong = {}
        frame_rays = synthetic.scene_rays(sc, path[0]).to(dev)                     # the same camera on every rank
        c4_idx = torch.randperm(N_RAYS, generator=torch.Generator().manual_seed(4))[:4096].to(dev)
        for name, rays_job in (("frame_512x640", frame_rays), ("c4_batch_4096_rays", frame_rays[c4_idx].contiguous())):
            n_job = rays_job.shape[0]
            job_frame = None
            if assemble == "peer":
                job_frame = mdist.PeerFrame(n_job, n_buffers=1)
            fn_band = (lambda r, sink=None: render(r, sink=sink))
            run = lambda: mdist.render_rays_sharded(rays_job, fn_band, frame=job_frame)
            for _ in range(3):
                run()
            barrier()
            reps = 10
            tot = 0.0
            for _ in range(reps):
                flush.zero_()
                a, b = ev(), ev()
                a.record(); out_rgb, out_depth = run(); b.record(); b.synchronize()
                tot += a.elapsed_time(b)
            ms = max_over_ranks(tot) / reps
            single_rgb, single_depth = render(rays_job)                             # this rank alone, whole job
            same = bool(torch.equal(out_rgb, single_rgb) and torch.equal(out_depth, single_depth))
            same = max_over_ranks(0.0 if same else 1.0) == 0.0
            strong[name] = {"value": n_job / (ms * 1e-3), "unit": "rays/s", "ms": ms, "rays": n_job,
                            "rays_per_gpu": n_job // world, "bit_equal_to_single_gpu": same}
            if job_frame is not None:
                job_frame.close()
        strong["api"] = "mvsnerf_b200.distributed.render_rays_sharded (" + \
            {"peer": "PeerFrame: kernel-epilogue NVLink peer stores + 1-element barrier",
             "nccl": "one NCCL all_gather_into_tensor of packed [n,4] pixels", "none": "single process"}[assemble] + ")"

        # ---- the other arithmetic tiers on the same workload (rank 0 reports; every rank runs the steps) ----------
        other = {}
        r32 = torch.empty_like(rgb); d32 = torch.empty_like(depth)
        rm = torch.empty_like(rgb); dm = torch.empty_like(depth)
        if rank == 0:
            t32 = min(ev_time(lambda: render(rays_dev[-1], lib.MLP_FP32, out=(r32, d32)), 2))
            render(rays_dev[-1], mode, out=(rm, dm))
            err = (rm - r32).abs()
            other["fp32_mode"] = {"value": N_RAYS / (t32 * 1e-3), "unit": "rays/s", "ms_per_frame": t32,
                                  "note": "MVSN_MLP_FP32 kernel (FFMA), the oracle-gated 1e-4 parity kernel"}
            other["parity_vs_fp32_kernel"] = {"rgb_linf": float(err.max()), "rgb_mse": float((err ** 2).mean()),
                                              "depth_linf": float((dm - d32).abs().max()),
                                              "gate": 5e-3 if args.mode in ("half", "pair") else 1e-4}
        if args.mode != "split" and not args.no_fp32_tier:
            # fp32 tier (north star: 1e-4 RGB Linf): MVSN_MLP_TC_SPLIT measured with the same rigour as the headline
            ms_s, kern_s, _ = timed_steps(lib.MLP_TC_SPLIT, 3, args.steps)
            e2e_s, _ = e2e_run(lib.MLP_TC_SPLIT, args.steps)
            if rank == 0:
                render(rays_dev[-1], lib.MLP_TC_SPLIT, out=(rm, dm))
                ks = sum(kern_s) / len(kern_s)
                tf = N_RAYS * FLOP_PER_RAY / (ks * 1e-3) / 1e12
                other["fp32_tier"] = {
                    "mlp_mode": "split", "dtype": MODE_DTYPE["split"], "value": world * N_RAYS / (ms_s * 1e-3),
                    "unit": "rays/s", "ms_per_step": ms_s,
                    "e2e": {"value": e2e_s, "unit": "rays/s", "h2d_bytes_per_step": hfr.h2d_bytes * world,
                            "d2h_bytes_per_step": hfr.d2h_bytes * world},
                    "roofline": {"bound": "tensor", "achieved": tf, "executed": 3 * tf * SPLIT_EXEC, "peak": pk["bf16_tflops"],
                                 "unit": "TFLOP/s", "frac": tf / pk["bf16_tflops"],
                                 "executed_frac": 3 * tf * SPLIT_EXEC / pk["bf16_tflops"],
                                 "kernel": MODE_KERNEL["split"], "kernel_ms": ks,
                                 "note": "achieved = algorithmic FLOPs of the reference MLP; executed = 3 MMAs per K-step on "
                                         "the kernel's own network (feature_linear folded into the views layer: 109 312 of "
                                         "the 125 696 MACs per sample)"},
                    "rgb_linf_vs_fp32_kernel": float((rm - r32).abs().max()), "gate": 1e-4,
                    "note": "MVSN_MLP_TC_SPLIT, the DEFAULT mode of backend.rendering / render_rays"}

        # ---- the north star's '>= 10x' denominator, measured in THIS run: the reference's PyTorch modules on this GPU ----
        ref_gpu = None
        if rank == 0 and world == 1 and not args.no_torch_gpu:
            ref_gpu = torch_gpu_reference(dev, vol, d, sc, rays_dev[-1])

    if rank == 0:
        tflops = N_RAYS * FLOP_PER_RAY / (kern * 1e-3) / 1e12
        gbs = N_RAYS * BYTES_PER_RAY / (kern * 1e-3) / 1e9
        prof = {}
        pj = os.path.join(ROOT, "profiles", "render_kernel_ncu.json")
        if os.path.exists(pj):
            prof = json.load(open(pj)).get(args.mode, {})
        par = "single GPU"
        if world > 1:
            par = (f"ray-sharded x{world}, volume replicated; frame assembly: " +
                   ("NVLink peer stores from the kernel epilogue into every rank's [n,4] frame + 1-element barrier per step"
                    if assemble == "peer" else "one NCCL all-gather of packed [n,4] pixels per step"))
        line = {
            "metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": MODE_DTYPE[args.mode], "data": "synthetic",
            "config": {"workload": "DTU-shaped 512x640 frame per GPU per step (configs[1]): 3 source views, pad 24, "
                                   "D=128 volume 8x128x176x208 resident, N_samples=128, ckpt mvsnerf-v0 weights",
                       "rays_per_gpu_per_step": N_RAYS, "mlp_mode": args.mode, "parallelism": par,
                       "l2": "flushed between timed steps (256 MiB write) and inputs (150 MB volume) exceed L2"},
            "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": hfr.h2d_bytes * world,
                    "d2h_bytes_per_step": hfr.d2h_bytes * world, "steps": args.steps,
                    "api": "mvsnerf_b200.backend.HostFrameRenderer.render -> mvsn_render_rays[_to_peers] (C ABI)"
                           + ("; frame assembly inside the loop" if world > 1 else "")},
            "gpu_launches": n_launch,
            "roofline": {"bound": "tensor", "achieved": tflops, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                         "frac": tflops / pk["bf16_tflops"], "traffic": prof.get("dram_bytes_per_launch"),
                         "traffic_source": prof.get("source"),
                         "kernel": MODE_KERNEL[args.mode], "kernel_ms": kern, "peak_source": pk["source"],
                         "frac_of_sustained_peak": tflops / pk["bf16_tflops_sustained"],
                         "hbm_gather_GBs": gbs, "hbm_frac": gbs / pk["hbm_gbs"],
                         "note": "algorithmic MLP FLOPs (32 178 176 / ray) over the render kernel's CUDA-event time on "
                                 "the timed steps' own launches, vs the measured cuBLAS bf16 burst peak; hbm_* is the "
                                 "51 248 B/ray gather definition (the kernel is tensor-bound, SURVEY 8(d))"},
            "volume_build": {"ms": t_build, "featurenet_ms": t_feat, "cost_volume_ms": t_cost, "costreg_ms": t_reg,
                             "cost_volume_GBs": (176.0 * nvox + 8.6e6) / (t_cost * 1e-3) / 1e9,
                             "cost_volume_hbm_frac": (176.0 * nvox + 8.6e6) / (t_cost * 1e-3) / 1e9 / pk["hbm_gbs"],
                             "costreg_TFLOPs": 111.3e9 / (t_reg * 1e-3) / 1e12,
                             "note": "once per scene (K-F FeatureNet + K-A cost volume + K-B CostRegNet, all hand-written kernels), "
                                     "not inside the step"},
            "strong_scaling": strong,
            "clocks": clocks, "wall_s_timed_region": t_wall,
        }
        if e2e_cam:
            line["e2e_camera"] = e2e_cam
        if trace:
            line["step_trace"] = trace
        if alt:
            line["assembly_comparison"] = alt
        if why:
            line["config"]["peer_store_fallback"] = why
        line.update(other)
        if ref_gpu:
            line["reference_pytorch_gpu"] = ref_gpu
            for k in ("value", "tf32_value"):
                line["reference_pytorch_gpu"][f"speedup_{k}_{args.mode}"] = value / ref_gpu[k]
                if "fp32_tier" in other:
                    line["reference_pytorch_gpu"][f"speedup_{k}_fp32_tier"] = other["fp32_tier"]["value"] / ref_gpu[k]
        if world == 1 and not args.no_finetune:
            try:
                line["finetune_step"] = finetune_step_bench(dev)
            except Exception as e:                                  # reported, never fatal for the headline
                line["finetune_step"] = {"error": f"{type(e).__name__}: {e}"}
        if world == 1 and not args.no_cpu_baseline:
            orc, _, weights, sc_cpu = cpu_reference_setup()
            sample = args.cpu_sample
            rays = rays_host[-1][torch.randperm(N_RAYS, generator=torch.Generator().manual_seed(0))[:sample]].contiguous()
            vol_cpu = vol.detach().cpu().contiguous()
            threads = cpu_pick_threads(orc, weights, sc_cpu, rays, vol_cpu)         # also the warm-up
            dt = cpu_render_sample(orc, weights, sc_cpu, rays, vol_cpu)
            line["cpu_baseline"] = {"value": sample / dt, "unit": "rays/s", "cores": threads,
                                    "host_cpus": os.cpu_count(), "kind": "port",
                                    "sample": f"{sample} random rays of one frame x 128 samples ({dt:.1f} s), oracle "
                                              f"port of the reference path, torch CPU, best of several pool sizes"}
        if last_frame is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, t in zip(("rgb", "depth"), last_frame):
                np.save(os.path.join(args.dump_outputs, name + ".npy"), t.cpu().numpy())
        print(json.dumps(line))
    if frame is not None:
        frame.close()
    if world > 1:
        dist.destroy_process_group()


def torch_gpu_reference(dev, vol, d, sc, rays):
    """The reference's own PyTorch path on this GPU (oracle modules on cuda, fp32, 5120-ray chunks as the notebooks use),
    one full 512x640 frame, with TF32 matmuls off (torch 2.x default) and on (torch-1.10's default, README.md:16)."""
    from oracle import mvsnerf_oracle as orc
    w = {k: v.to(dev) for k, v in orc.load_weights_npz(WEIGHTS).items()}
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    out = {"unit": "rays/s", "rays": N_RAYS, "chunk": 5120}
    try:
        for key, tf32 in (("value", False), ("tf32_value", True)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.allow_tf32 = tf32
            with torch.no_grad():
                orc.render_rays(rays[:10240], vol, d.imgs_raw, d.pose_source, w, H, W, sc.near_far, float(PAD), n_samples=S,
                                chunk=5120)
                torch.cuda.synchronize()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                orc.render_rays(rays, vol, d.imgs_raw, d.pose_source, w, H, W, sc.near_far, float(PAD), n_samples=S, chunk=5120)
                b.record(); b.synchronize()
            out[key] = N_RAYS / (a.elapsed_time(b) * 1e-3)
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    out["note"] = ("oracle restatement of the reference's PyTorch modules on this B200 (library kernels: cuBLAS/cuDNN/"
                   "grid_sample), one full frame, measured in this run; the north star's >=10x denominator")
    return out


def finetune_step_bench(dev):
    """BASELINE config 3 shape: one fine-tuning step = 1024 rays x 128 samples against an 8x128x200x200 RefVolume
    (800x800 Blender-shaped, pad 0, white_bkgd), forward + backward + Adam on MLP and volume
    (train_mvs_nerf_finetuning_pl.py:140-189), through backend.rendering under autograd."""
    from mvsnerf_b200 import backend, synthetic
    if not hasattr(backend, "finetune_step_timing"):
        return {"error": "backend.finetune_step_timing not available in this build"}
    return backend.finetune_step_timing(dev, WEIGHTS)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default=os.environ.get("MVSN_BENCH_MODE", "pair"), choices=["fp32", "half", "split", "pair"],
                    help="MLP arithmetic of the headline: pair = tcgen05 CTA-pair kernel (5e-3 tier, default); "
                         "split = fp32-grade tensor mode (also always reported as fp32_tier); half = round-1 kernel")
    ap.add_argument("--assemble", default=os.environ.get("MVSN_BENCH_ASSEMBLE", "peer"), choices=["peer", "nccl"],
                    help="N > 1: kernel-epilogue NVLink peer stores (falls back to nccl when peers cannot be mapped) or "
                         "one NCCL all-gather per step")
    ap.add_argument("--cpu-sample", type=int, default=8192)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fp32-tier", action="store_true")
    ap.add_argument("--no-torch-gpu", action="store_true")
    ap.add_argument("--no-finetune", action="store_true")
    ap.add_argument("--no-assembly-comparison", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's rgb and depth as DIR/rgb.npy, DIR/depth.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.gpus != 1):
        ap.error("--dump-outputs writes the frame of a single-GPU run of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
