#!/usr/bin/env python
"""bench.py -- rays/sec of the SceneRF ray-render hot path on B200 (BASELINE.json metric), one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload B|A|C] [--precision fp16|fp32]
                    [--dump-outputs DIR]

A "step" is one full render_rays_batch-equivalent pass (gaussian proposal MLP, sampling+sort, main MLP, compositing,
RaySOM skipped as inference callers do, multi-GPU gather) over every ray of the workload:
  workload B (default, BASELINE.json configs[1]): KITTI 1226x370 full-frame novel view, 453 620 rays x 128 samples.
Features and weights are packed and resident before the timed region (SURVEY.md 8d).  `value` times the device-resident
call; `e2e` times the reference-facing host-buffer call (pinned pixels H2D + depth/rgb D2H inside the timed region).
N > 1 (torchrun): frame-per-GPU layout -- every rank renders its own full frame (own pose) and the packed depth+rgb
of all frames are all-gathered over NCCL; per-GPU work is fixed => "scaling": "weak".
--dump-outputs DIR writes what the last timed step returned.  Inputs, weights and noise seeds depend only on the
arguments, so two builds run with the same arguments can be compared array by array.
--impl reference times the CPU restatement of the reference (oracle/, pinned to the reference's own outputs) on the host
cores with a process pool; the reference itself is PyTorch-on-Python and is not present on the GPU box.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
if "reference" in sys.argv:
    # torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core (set before numpy loads BLAS)
    for _k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ.pop(_k, None)

import numpy as np  # noqa: E402

FLOP_MAIN = 2 * 5405696       # per main sample point  (BASELINE.md section 3)
FLOP_GAUSS = 2 * 5404672      # per gaussian-proposal point


def workload(name):
    from scenerf_b200 import synth
    if name == "A":
        cfg = synth.config_A()
        pix = synth.random_pixels(1, 1024, cfg.img_W, cfg.img_H)
        desc = "A: KITTI single image, 1024 rays x 64 samples"
    elif name == "C":
        cfg = synth.config_C()
        pix = synth.grid_pixels(cfg.img_W, cfg.img_H)
        desc = "C: BundleFusion 640x480 full frame, 307200 rays x 96 samples"
    elif name == "Bp":
        cfg = synth.config_B(name="Bp", sphere_W=1500, sphere_H=452)
        pix = synth.grid_pixels(cfg.img_W, cfg.img_H)
        desc = "B': config B's frame (453620 rays x 128 samples) over the reference-default 1500x452 sphere grid (420 MB pyramid)"
    else:
        cfg = synth.config_B()
        pix = synth.grid_pixels(cfg.img_W, cfg.img_H)
        desc = "B: KITTI 1226x370 full-frame novel view, 453620 rays x 128 samples"
    return cfg, np.ascontiguousarray(pix), desc


def hp_from_cfg(cfg):
    v_min, v_max, h_min, h_max = cfg.angles()
    return dict(dataset=cfg.dataset, n_pts_uni=cfg.n_pts_uni, n_gaussians=cfg.n_gaussians,
                n_pts_per_gaussian=cfg.n_pts_per_gaussian, std=cfg.std, max_sample_depth=cfg.max_sample_depth,
                out_img_W=cfg.sphere_W, out_img_H=cfg.sphere_H, som_sigma=cfg.som_sigma, v_angle_min=v_min,
                v_angle_max=v_max, h_angle_min=h_min, h_angle_max=h_max)


def flop_per_ray(cfg):
    return cfg.S * FLOP_MAIN + cfg.n_gaussians * FLOP_GAUSS


# ------------------------------------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
# CPU arm.  Preferred: the reference's OWN class (oracle/_ref, staged by oracle/build_ref.py from the unmodified
# reference sources) run through the SURVEY 8c shim on all host threads torch gives it -> kind "reference".
# Fallback when oracle/_ref is absent: the numpy restatement (oracle/scenerf_oracle.py) with a fork pool -> kind "port".
# ------------------------------------------------------------------------------------------------------------------
_CPU = {}


def _cpu_init(cfg, pyr_seed, blas_threads):
    from threadpoolctl import threadpool_limits
    from oracle.scenerf_oracle import OracleRenderer   # checker / CPU baseline only
    from scenerf_b200 import synth
    _CPU["limit"] = threadpool_limits(limits=blas_threads)
    pm, pg = synth.make_model_params(cfg)
    _CPU["r"] = OracleRenderer(cfg, pm, pg)
    _CPU["cfg"] = cfg


def _cpu_chunk(args):
    pix, seed = args
    cfg = _CPU["cfg"]
    rng = np.random.default_rng(seed)
    nu = rng.random((pix.shape[0], cfg.n_pts_uni), dtype=np.float32)
    nn_ = rng.standard_normal((pix.shape[0], cfg.n_gaussians * cfg.n_pts_per_gaussian)).astype(np.float32)
    out = _CPU["r"].render_rays_batch(cfg.K, cfg.T, _CPU["pyr"], pix, pix.shape[0], nu, nn_)
    return float(out["depth"].sum())


def cpu_port_rays_per_sec(cfg, pix, pyramid, target_seconds=15.0, chunk=128):
    """Fallback arm: the numpy oracle on a bounded sample of the workload's rays, fork pool over ray chunks with a
    FIXED layout (16 workers x cores/16 BLAS threads) so that boxes with the same core count agree."""
    import multiprocessing as mp
    cores = effective_cpus()[0]
    workers = max(1, min(16, cores // 2))
    blas = max(1, cores // workers)
    _CPU["pyr"] = pyramid                      # inherited by fork (copy-on-write, no pickling of 281 MB)
    ctx = mp.get_context("fork")
    with ctx.Pool(workers, initializer=_cpu_init, initargs=(cfg, 0, blas)) as pool:
        rng = np.random.default_rng(0)
        sel = rng.permutation(pix.shape[0])
        mk = lambda i: (np.ascontiguousarray(pix[sel[(i * chunk + np.arange(chunk)) % sel.shape[0]]]), i)
        t0 = time.perf_counter()
        pool.map(_cpu_chunk, [mk(i) for i in range(workers)])            # warm-up + calibration round
        t_round = time.perf_counter() - t0
        rounds = int(max(1, min(20, target_seconds / max(t_round, 1e-3))))
        n_chunks = workers * rounds
        t0 = time.perf_counter()
        pool.map(_cpu_chunk, [mk(workers + i) for i in range(n_chunks)])
        dt = time.perf_counter() - t0
    n_rays = n_chunks * chunk
    return n_rays / dt, dict(cores=workers * blas, kind="port",
                             sample="%d rays x %d samples of the workload (random subset, %d-ray chunks, %d procs x %d BLAS threads), %.1f s"
                                    % (n_rays, cfg.S, chunk, workers, blas, dt))


# Fixed layout of the reference CPU arm, chosen by tools/ref_probe.py on the B200 box's host (2 x 32-core Xeon 8562Y+,
# 128 logical CPUs; profiles/r2_reference_cpu_layout_probe.log): ONE process with 64-128 intra-op threads reaches only
# 35-300 rays/s (the reference's chain of small ops does not scale past ~16 threads), 8 processes x 16 threads reach
# 800-950 rays/s.  So the arm is 8 worker processes, each running the reference's own class on its own rays.
REF_PROCS = 8
REF_RAYS_PER_PROC = 512          # rays per reference call (one chunk): 8 x 512 = 4096 rays per step


def _ref_worker_main(conn, workload_name, threads, seed):
    """Worker process: builds the reference model + its own copy of the synthetic pyramid, then serves 'step' requests."""
    try:
        for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
            os.environ.pop(k, None)
        import torch
        torch.set_num_threads(threads)
        from oracle import ref_runner
        cfg, pix, _ = workload(workload_name)
        tm = ref_runner.ReferenceTimer(cfg, pix, make_cpu_pyramid(cfg), threads=threads, seed=seed)
        conn.send(("ready", tm.threads))
        while True:
            msg = conn.recv()
            if msg[0] == "stop":
                break
            conn.send(("done", tm.step(msg[1])))
    except Exception as e:          # report instead of hanging the parent
        conn.send(("error", repr(e)))


def effective_cpus():
    """CPUs this process may really use: min(logical CPUs, scheduler affinity, cgroup CPU quota).  A GPU lease can be a
    container with a CPU quota far below os.cpu_count() (the 1-GPU and 8-GPU boxes of this pool differ 3x in what the same
    128-thread layout achieves); running more threads than the quota only oversubscribes."""
    n = os.cpu_count() or 1
    info = {"logical": n}
    try:
        aff = len(os.sched_getaffinity(0))
        info["affinity"] = aff
        n = min(n, aff)
    except Exception:
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                txt = f.read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    q = float(txt[0]) / float(txt[1])
                    info["cgroup_quota"] = q
                    n = min(n, max(1, int(q + 0.5)))
            else:
                q = float(txt[0])
                if q > 0:
                    with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f2:
                        q /= float(f2.read().split()[0])
                    info["cgroup_quota"] = q
                    n = min(n, max(1, int(q + 0.5)))
            break
        except Exception:
            continue
    try:
        info["loadavg_1min"] = os.getloadavg()[0]
    except Exception:
        pass
    info["effective"] = n
    return n, info


class ReferencePool:
    """REF_PROCS processes x (host threads / REF_PROCS) torch threads, each timing the reference's own
    SceneRF.render_rays_batch (oracle/_ref) on disjoint random rays of the workload."""

    def __init__(self, workload_name):
        import multiprocessing as mp
        from oracle import ref_runner
        self.ok = ref_runner.available()
        if not self.ok:
            return
        cores, self.cpu_info = effective_cpus()
        self.procs = max(1, min(REF_PROCS, cores // 2))
        self.threads = max(1, cores // self.procs)
        ctx = mp.get_context("spawn")
        self.workers = []
        for i in range(self.procs):
            parent, child = ctx.Pipe()
            pr = ctx.Process(target=_ref_worker_main, args=(child, workload_name, self.threads, i), daemon=True)
            pr.start()
            self.workers.append((pr, parent))
        for _, c in self.workers:
            tag, val = c.recv()
            if tag != "ready":
                raise RuntimeError("reference worker failed: %s" % (val,))

    def step(self, n_rays):
        """All workers run one reference call of n_rays rays concurrently; -> (wall seconds, per-worker seconds)."""
        t0 = time.perf_counter()
        for _, c in self.workers:
            c.send(("step", n_rays))
        per = []
        for _, c in self.workers:
            tag, val = c.recv()
            if tag != "done":
                raise RuntimeError("reference worker failed: %s" % (val,))
            per.append(val)
        return time.perf_counter() - t0, per

    def close(self):
        for pr, c in self.workers:
            try:
                c.send(("stop",))
            except Exception:
                pass
        for pr, _ in self.workers:
            pr.join(timeout=10)


def cpu_baseline(workload_name, cfg, pix, pyramid, target_seconds=20.0):
    """The bounded CPU sample of the default arm (rank 0, N=1 only): a few pool steps of the reference, ~target_seconds."""
    from oracle import ref_runner
    pool = ReferencePool(workload_name)
    if not pool.ok:
        v, info = cpu_port_rays_per_sec(cfg, pix, pyramid, target_seconds=target_seconds)
        return {"value": v, "unit": "rays/s", "cores": info["cores"], "kind": "port", "sample": info["sample"]}
    try:
        n = min(REF_RAYS_PER_PROC, pix.shape[0])
        t_warm, _ = pool.step(n)
        times = []
        while sum(times) < target_seconds - t_warm and len(times) < 6:
            times.append(pool.step(n)[0])
        v = n * pool.procs * len(times) / sum(times)
        return {"value": v, "unit": "rays/s", "cores": pool.procs * pool.threads, "kind": "reference", "cpu_model": ref_runner.cpu_model_name(),
                "cpus": pool.cpu_info,
                "sample": "%d steps; each step = %d concurrent calls (one per process, %d torch threads each) of the reference's "
                          "SceneRF.render_rays_batch (oracle/_ref) on %d random rays x %d samples of the workload in one chunk; %.1f s after a %.1f s warm-up step"
                          % (len(times), pool.procs, pool.threads, n, cfg.S, sum(times), t_warm)}
    finally:
        pool.close()


def make_cpu_pyramid(cfg, seed=5):
    rng = np.random.default_rng(seed)
    from scenerf_b200 import synth
    return {k: (rng.standard_normal((c, h, w), dtype=np.float32) * np.float32(0.5))
            for k, (c, h, w) in zip(synth.SCALE_KEYS, synth.pyramid_shapes(cfg.sphere_W, cfg.sphere_H))}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on this box's host cores.  One step = REF_PROCS
    concurrent render_rays_batch calls (one per worker process, REF_RAYS_PER_PROC rays each, one chunk) on a bounded sample
    of the workload's rays."""
    if rank != 0:
        return
    from oracle import ref_runner
    cfg, pix, desc = workload(args.workload)
    pool = ReferencePool(args.workload)
    if pool.ok:
        try:
            n = min(REF_RAYS_PER_PROC, pix.shape[0])
            for _ in range(max(1, min(args.warmup, 2))):
                pool.step(n)
            times = [pool.step(n)[0] for _ in range(args.steps)]
        finally:
            pool.close()
        value = n * pool.procs * len(times) / sum(times)
        ms = float(np.mean(times)) * 1e3
        cpu = {"value": value, "unit": "rays/s", "cores": pool.procs * pool.threads, "kind": "reference", "cpu_model": ref_runner.cpu_model_name(),
               "cpus": pool.cpu_info,
               "sample": "each step = %d concurrent calls (one per process, %d torch threads each) of the reference's SceneRF.render_rays_batch "
                         "(unmodified sources in oracle/_ref through the SURVEY 8c shim) on %d random rays x %d samples of the workload in one chunk; "
                         "step times min/median/max %.2f/%.2f/%.2f s; layout fixed by profiles/r2_reference_cpu_layout_probe.log"
                         % (pool.procs, pool.threads, n, cfg.S, min(times), float(np.median(times)), max(times))}
        what = "the reference's own SceneRF class (unmodified sources staged in oracle/_ref) on host cores"
        rays_per_step = n * pool.procs
    else:
        pyr = make_cpu_pyramid(cfg)
        vals, info = [], None
        for i in range(args.warmup + args.steps):
            v, info = cpu_port_rays_per_sec(cfg, pix, pyr, target_seconds=4.0)
            if i >= args.warmup:
                vals.append(v)
        value, ms = float(np.mean(vals)), None
        cpu = {"value": value, "unit": "rays/s", "cores": info["cores"], "kind": "port", "sample": info["sample"]}
        what = "CPU restatement of the reference (oracle/, numpy+BLAS) on host cores -- oracle/_ref not staged"
        rays_per_step = None
    line = {"metric": "rays/sec", "value": value, "unit": "rays/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": desc, "what": what, "rays_per_step": rays_per_step, "samples_per_ray": cfg.S},
            "cpu_baseline": cpu,
            "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
def run_sweep(args, rank, world, local):
    """--workload sweep: the reconstruction rows (SURVEY 8f-2 TSDF integrate, 8f-4 novel-view sweep).  One "step" = the
    sweep of one source frame with the defaults of generate_novel_depths.py / depth2tsdf.py: 1220x370 image, stride 2,
    63 poses, 64 samples per ray, 256x256x32 TSDF volume; with N GPUs the poses are sharded and the volumes merged.
    Not the headline metric: a second JSON line format with the TSDF kernel's HBM roofline and the reference's CPU TSDF
    path (oracle restatement) timed beside it."""
    import time
    import torch
    import torch.distributed as dist
    from scenerf_b200 import synth, sweep
    from scenerf_b200.renderer import B200Renderer
    from scenerf_b200.tsdf import TSDFVolume
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    cfg = synth.config_A(name="sweep")                     # KITTI class defaults: 64 samples/ray, sphere 1500x452
    pm, pg = synth.make_model_params(cfg)
    to = lambda d: {k: torch.from_numpy(v) for k, v in d.items()}
    # the sweep renders 63 poses of ONE source frame: the per-image latent table (built once, first call) is the natural mode
    r = B200Renderer(hp_from_cfg(cfg), to(pm), to(pg), device=dev, precision=args.precision, preproject=bool(args.sweep_table))
    x_rgb = {k: torch.from_numpy(v).to(dev) for k, v in synth.make_pyramid(3, cfg.sphere_W, cfg.sphere_H).items()}
    cam_K = torch.from_numpy(synth.KITTI_K).to(dev)
    sw = sweep.NovelDepthSweep(r, cam_K, x_rgb, img_size=(1220, 370), scale=args.sweep_scale)
    poses = dict(list(sweep.sample_rel_poses(step=0.5, angle=10, max_distance=10.1).items())[:args.sweep_poses])
    T_velo2cam = np.array([[0.0, -1.0, 0.0, 0.0], [0.0, 0.0, -1.0, -0.08], [1.0, 0.0, 0.0, -0.27], [0, 0, 0, 1.0]])
    vol_bnds = np.zeros((3, 2))
    vol_bnds[:, 0] = [0, -25.6, -2]
    vol_bnds[:, 1] = vol_bnds[:, 0] + [51.2, 51.2, 6.4]

    def frame():
        return sw.reconstruct(poses, T_velo2cam, vol_bnds, voxel_size=0.2, rank=rank, world=world)

    for _ in range(args.warmup):
        vol = frame()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sw.launches = 0
    e0.record()
    for _ in range(args.steps):
        vol = frame()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())

    # --- the TSDF kernel alone, against HBM ------------------------------------------------------------------------
    depth, rgb = sw.render(list(poses.values())[1].to(cam_K), sweep.COLOR_PNG)
    tv = TSDFVolume(vol_bnds, voxel_size=0.2, device=dev)
    pose = np.linalg.inv(T_velo2cam) @ list(poses.values())[1].numpy().astype(np.float64)
    n_it = 200
    for _ in range(5):
        tv.integrate(rgb, depth, synth.KITTI_K, pose)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n_it):
        tv.integrate(rgb, depth, synth.KITTI_K, pose)
    e1.record()
    torch.cuda.synchronize()
    tsdf_us = e0.elapsed_time(e1) / n_it * 1e3
    n_vox = int(np.prod(tv._vol_dim))
    touched = float((tv.get_weight() > 0).mean())
    # algorithmic bytes per launch: every voxel is projected (no memory), touched voxels read tsdf+weight (8 B), write
    # weight (4 B) and, when the new observation wins (all of them on a repeat of the same frame), tsdf+colour (8 B),
    # plus the depth/colour pixel (16 B, L2-resident image of 7.2 MB counted once)
    alg_bytes = n_vox * touched * (8 + 4 + 8) + depth.numel() * 16
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm = float(peaks.get("hbm_gbs") or 6500.0)

    out = {"metric": "sweep frames/sec (one source frame: %d poses rendered at stride %d + TSDF fusion)" % (len(poses), args.sweep_scale),
           "value": 1e3 / ms, "unit": "frames/s", "ms_per_frame": ms, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "rays_per_pose": int(sw.pixels.shape[0]), "samples_per_ray": cfg.S, "poses": len(poses), "precision": args.precision,
           "latent_table": bool(args.sweep_table),
           "rays_per_sec": len(poses) * int(sw.pixels.shape[0]) / (ms * 1e-3), "gpu_launches": sw.launches // max(1, args.steps),
           "volume": [int(d) for d in tv._vol_dim], "volume_touched_frac": float((vol.get_weight() > 0).mean()),
           "tsdf_kernel": {"us_per_launch": tsdf_us, "algorithmic_bytes": alg_bytes, "achieved_gbps": alg_bytes / (tsdf_us * 1e-6) / 1e9,
                           "peak_gbps": hbm, "frac": alg_bytes / (tsdf_us * 1e-6) / 1e9 / hbm, "touched_frac": touched,
                           "note": "includes the host-side 4x4 inverse + ctypes call of TSDFVolume.integrate; 2.1 M voxels is launch-latency bound"}}
    if rank == 0 and not args.no_cpu_baseline:
        from oracle.tsdf_oracle import TSDFVolumeOracle
        ov = TSDFVolumeOracle(vol_bnds, 0.2, 10)
        d_np, c_np = depth.cpu().numpy(), rgb.cpu().numpy()
        t0 = time.perf_counter()
        for _ in range(3):
            ov.integrate(c_np, d_np, synth.KITTI_K, pose, 1.0)
        out["tsdf_cpu_baseline"] = {"ms_per_integrate": (time.perf_counter() - t0) / 3 * 1e3, "kind": "port", "cores": 1,
                                    "sample": "3 integrations of one 1220x370 frame into the 256x256x32 volume (numpy restatement of fusion.py CPU path)"}
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def run_train(args, rank, world, local):
    """--workload train: the backward row (SURVEY 8f-1).  One step = what the reference's training does per source frame
    (scenerf.py:243-320): render_rays_batch on 1200 random pixels of the stride-2 grid in ONE chunk (64 samples/ray, KITTI
    defaults, sphere 1500x452), a depth + colour + KL loss, backward to the 2x22 ResnetFC tensors and the 5 feature maps.
    float32 SIMT forward + backward (csrc/backward.cu).  Every rank runs its own frame (data parallel; the gradient
    all-reduce stays PyTorch DDP's, SURVEY 8e)."""
    import time
    import torch
    import torch.distributed as dist
    from scenerf_b200 import synth
    from scenerf_b200.autograd import TrainableRenderer, PARAM_KEYS
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = synth.config_A(name="train")
    R = args.rays if args.rays > 0 else 1200
    pm, pg = synth.make_model_params(cfg)
    mk = lambda d: {k: torch.from_numpy(d[k]).to(dev).requires_grad_(True) for k in PARAM_KEYS}
    tm, tg = mk(pm), mk(pg)
    x_rgb = {k: torch.from_numpy(v).to(dev).requires_grad_(True) for k, v in synth.make_pyramid(5 + rank, cfg.sphere_W, cfg.sphere_H).items()}
    t = TrainableRenderer(hp_from_cfg(cfg), tm, tg, device=dev, rng="philox", matmul=args.train_matmul)
    K, T = torch.from_numpy(cfg.K).to(dev), torch.from_numpy(cfg.T).to(dev)
    grid = synth.grid_pixels(cfg.img_W, cfg.img_H, stride=2)
    sel = np.random.default_rng(7 + rank).permutation(grid.shape[0])[:R]
    pix_host = torch.from_numpy(np.ascontiguousarray(grid[sel])).pin_memory()
    target = torch.rand(R, 3, device=dev)

    def step():
        for p_ in list(tm.values()) + list(tg.values()) + list(x_rgb.values()):
            p_.grad = None
        out = t.render_rays_batch(K, T, x_rgb, sampled_pixels=pix_host.to(dev, non_blocking=True), ray_batch_size=R)
        loss = (out["color"] - target).abs().mean() + 0.01 * out["depth"].mean() + out["loss_kl"].mean() \
            + 0.01 * (out["gaussian_means"] - out["depth"].detach().unsqueeze(-1)).abs().min(dim=1)[0].mean()
        loss.backward()
        return loss

    for _ in range(args.warmup):
        loss = step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    e[0].record()
    for _ in range(args.steps):
        loss = step()
        lv = float(loss.detach().cpu())                       # D2H read of the step's result
    e[1].record()
    torch.cuda.synchronize()
    ms = e[0].elapsed_time(e[1]) / args.steps
    if world > 1:
        tt = torch.tensor([ms], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    # forward / backward split (CUDA events around the two halves of one more step)
    for p_ in list(tm.values()) + list(tg.values()) + list(x_rgb.values()):
        p_.grad = None
    e[2].record()
    out = t.render_rays_batch(K, T, x_rgb, sampled_pixels=pix_host.to(dev), ray_batch_size=R)
    loss = (out["color"] - target).abs().mean() + 0.01 * out["depth"].mean() + out["loss_kl"].mean()
    e[3].record()
    loss.backward()
    e[0].record()
    torch.cuda.synchronize()
    fwd_ms, bwd_ms = e[2].elapsed_time(e[3]), e[3].elapsed_time(e[0])
    flop_fwd = R * flop_per_ray(cfg)
    flop_step = 4.0 * flop_fwd          # forward + recompute + dX GEMMs + dW GEMMs, each = one forward's FLOPs
    fp32_peak = 148 * 128 * 2 * 1.965e9 / 1e12          # 148 SMs x 128 FMA lanes x 2 x max clock
    bound = "fp32 FMA (SIMT)"
    if args.train_matmul == "tf32":
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        fp32_peak = float(peaks.get("bf16_tflops_sustained") or 1400.0) / 2.0      # kind::tf32 issues at half the kind::f16 rate
        bound = "tensor (tcgen05 kind::tf32; peak = measured bf16 sustained / 2)"
    res = {"metric": "training rays/sec (render_rays_batch forward + backward, %d rays x %d samples per step)" % (R, cfg.S),
           "value": world * R / (ms * 1e-3), "unit": "rays/s", "ms_per_step": ms, "n_gpus": world, "steps": args.steps,
           "warmup": args.warmup, "dtype": "f32" if args.train_matmul == "fp32" else "tf32 operands, f32 storage and accumulate",
           "data": "synthetic", "scaling": "weak", "higher_is_better": True,
           "forward_ms": fwd_ms, "backward_ms": bwd_ms, "loss": lv,
           "gpu_launches": int(t.renderer.last_launches + t.renderer.last_backward_launches),
           "roofline": {"bound": bound, "achieved": 3.0 * flop_fwd / (ms * 1e-3) / 1e12, "peak": fp32_peak, "unit": "TFLOP/s",
                        "frac": 3.0 * flop_fwd / (ms * 1e-3) / 1e12 / fp32_peak,
                        "algorithmic_flop_per_step": 3.0 * flop_fwd, "dense_flop_per_step_with_recompute": flop_step,
                        "note": "ALGORITHMIC flops (forward + dX + dW of the dense 2480-wide latent) / time; SIMT peak = 148 SMs x 128 lanes x "
                                "2 FLOP x 1.965 GHz.  Not a utilisation figure: the lin_z K-segments of pyramid scales that no point of a "
                                "chunk reaches (exact zeros, quirk Q2; typically 2240 of the 2480 latent columns) are skipped on the "
                                "device, and the backward recomputes the forward per 9472-point chunk"}}
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import scenerf_oracle as so, backward_oracle as bo
        n = 24
        orc = so.OracleRenderer(cfg, pm, pg)
        pyr = synth.make_pyramid(5, cfg.sphere_W, cfg.sphere_H)
        rng = np.random.default_rng(0)
        nu, nn_ = rng.random((n, cfg.n_pts_uni)).astype(np.float32), rng.standard_normal((n, cfg.n_gaussians * cfg.n_pts_per_gaussian)).astype(np.float32)
        cot = {"depth": np.full(n, 0.01 / n), "color": np.full((n, 3), 1.0 / (3 * n)), "loss_kl": np.full(n, 1.0 / n)}
        t0 = time.perf_counter()
        bo.render_backward(orc, cfg.K, cfg.T, pyr, grid[sel][:n], nu, nn_, cot)
        dt = time.perf_counter() - t0
        res["cpu_baseline"] = {"value": n / dt, "unit": "rays/s", "cores": os.cpu_count(), "kind": "port",
                               "sample": "%d rays x %d samples forward + backward with the numpy oracle (BLAS threads), %.1f s" % (n, cfg.S, dt)}
    if rank == 0:
        print(json.dumps(res))
    if world > 1:
        dist.destroy_process_group()


def run_lattice(args, rank, world, local):
    """--workload E: density-only query of the 256^3 lattice (SURVEY 8d config E; scenerf.py:505-547 `predict`), z-slab per GPU
    + all-gather of the densities.  One step = the whole lattice (16.78 M points, 181.4 TFLOP)."""
    import time
    import torch
    import torch.distributed as dist
    from scenerf_b200 import synth, lattice
    from scenerf_b200.renderer import B200Renderer
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = synth.config_A(name="lattice")
    pm, pg = synth.make_model_params(cfg)
    to = lambda d: {k: torch.from_numpy(v) for k, v in d.items()}
    r = B200Renderer(hp_from_cfg(cfg), to(pm), to(pg), device=dev, precision=args.precision)
    x_rgb = {k: torch.from_numpy(v).to(dev) for k, v in synth.make_pyramid(5, cfg.sphere_W, cfg.sphere_H).items()}
    K = torch.from_numpy(cfg.K).to(dev)
    run = lambda: lattice.density_lattice(r, x_rgb, K, rank=rank, world=world)
    for _ in range(args.warmup):
        d = run()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        d = run()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    if world > 1:
        tt = torch.tensor([ms], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    n_pts = 256 ** 3
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("bf16_tflops_sustained") or 1400.0)
    res = {"metric": "lattice points/sec (density query of the 256^3 lattice)", "value": n_pts / (ms * 1e-3), "unit": "points/s",
           "ms_per_step": ms, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "dtype": args.precision, "data": "synthetic",
           "scaling": "strong", "higher_is_better": True, "gpu_launches": int(r.last_lattice_launches),
           "density_mean": float(d.mean()), "density_in_image_frac": float((d > 0).float().mean()),
           "roofline": {"bound": "tensor", "achieved": n_pts * FLOP_MAIN / (ms * 1e-3) / 1e12, "peak": peak, "unit": "TFLOP/s",
                        "frac": n_pts * FLOP_MAIN / (ms * 1e-3) / 1e12 / peak, "note": "whole step incl. point generation and z-slab all-gather"}}
    if rank == 0 and not args.no_cpu_baseline:
        from oracle.scenerf_oracle import OracleRenderer
        orc = OracleRenderer(cfg, pm, pg)
        pyr = synth.make_pyramid(5, cfg.sphere_W, cfg.sphere_H)
        xa = lattice.axis(*lattice.DEFAULT_X, "cpu").numpy(); ya = lattice.axis(*lattice.DEFAULT_Y, "cpu").numpy()
        za = lattice.axis(*lattice.DEFAULT_Z, "cpu").numpy()
        ncol = 32
        pts = np.zeros((ncol, 256, 3), np.float32)
        pts[:, :, 0] = xa[100:100 + ncol, None]; pts[:, :, 1] = ya[128]; pts[:, :, 2] = za[None, :]
        t0 = time.perf_counter()
        orc.predict(orc.pm, pts, pyr, cfg.K, np.tile(np.float32([[0, 0, 1]]), (ncol, 1)))
        dt = time.perf_counter() - t0
        res["cpu_baseline"] = {"value": ncol * 256 / dt, "unit": "points/s", "cores": os.cpu_count(), "kind": "port",
                               "sample": "%d columns x 256 points with the numpy oracle (BLAS threads), %.1f s" % (ncol, dt)}
    if rank == 0:
        print(json.dumps(res))
    if world > 1:
        dist.destroy_process_group()


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


PREC_DESC = {"fp32tc": "fp32-grade on tensor cores: fp16 hi/lo split operands (22 mantissa bits), fp32 accumulate in TMEM (tcgen05 kind::f16, 4 partial products)",
             "fp16": "fp16 operands, fp32 accumulate (tcgen05 kind::f16) -- reduced-precision fast mode",
             "fp32": "fp32 SIMT FMA"}
PREC_DTYPE = {"fp32tc": "fp32 (2 x fp16 split operands, fp32 accumulate)", "fp16": "fp16", "fp32": "f32"}


def time_loop(fn, steps, warmup, sync):
    """warmup untimed calls, then `steps` calls between CUDA events on the current stream; -> ms per call."""
    import torch
    for _ in range(warmup):
        fn()
    sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    sync()
    return e0.elapsed_time(e1) / steps


DUMP_LIMIT_BYTES = 64 * 10 ** 6
NPY_HEADER_BYTES = 128


def dump_outputs(path, arrays, ray_axis=0, limit_bytes=DUMP_LIMIT_BYTES, seed=0):
    """--dump-outputs: every array of `arrays` (name -> tensor, rays along `ray_axis`) as path/<name>.npy in float32, so
    that two builds can be compared output for output.  Above `limit_bytes` in all, every array keeps the same fixed,
    seeded sample of rays (in ray order), whose indices are written as path/ray_index.npy (float64)."""
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    n = next(iter(arrays.values())).shape[ray_axis]
    per_ray = sum(a.nbytes for a in arrays.values()) // max(1, n)
    budget = limit_bytes - NPY_HEADER_BYTES * (len(arrays) + 1)
    if per_ray * n > budget:
        keep = min(n, budget // (per_ray + 8))
        idx = np.sort(np.random.default_rng(seed).choice(n, keep, replace=False))
        arrays = {k: np.take(a, idx, axis=ray_axis) for k, a in arrays.items()}
        arrays["ray_index"] = idx.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), np.ascontiguousarray(a))


def max_over_ranks(ms, dev, world):
    import torch
    import torch.distributed as dist
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def measure_workload_D(args, rank, world, dev, sync, mk_renderer):
    """BASELINE.json configs[3] (SURVEY 8d config D; reference caller: save_depth_metrics.py:105-118): 8 independent frames
    (8 feature pyramids, poses t_z = 1..8 m), 16 384 integer LiDAR-like pixels each, 64 samples/ray.  One step = all 8 frames
    rendered and the packed depth+rgb of every frame present on every rank.  Both layouts of SURVEY 8e are timed:
      frame-per-GPU : frame f on rank f % N, one all-gather of the finished frames;
      ray-sharded   : every frame's rays split in N contiguous ranges (every rank holds all 8 packed pyramids)."""
    import torch
    import torch.distributed as dist
    from scenerf_b200 import synth
    from scenerf_b200 import dist as sdist
    n_frames, n_pix = 8, 16384
    cfgs = [synth.config_A(name="D%d" % f, tz=float(f + 1)) for f in range(n_frames)]
    rng = np.random.default_rng(17)
    pix = [torch.from_numpy(np.stack([rng.integers(0, cfgs[0].img_W, n_pix), rng.integers(0, cfgs[0].img_H, n_pix)], 1).astype(np.float32)).to(dev)
           for _ in range(n_frames)]
    K = torch.from_numpy(cfgs[0].K)
    Ts = [torch.from_numpy(c.T) for c in cfgs]
    mine = [f for f in range(n_frames) if f % world == rank]
    need = list(range(n_frames)) if world > 1 else mine          # ray-sharded layout: all pyramids on every rank
    rend, x_rgbs = {}, {}
    for f in need:
        gen = torch.Generator(device=dev)
        gen.manual_seed(100 + f)
        x_rgbs[f] = {k: torch.randn((c, h, w), generator=gen, device=dev) * 0.5
                     for k, (c, h, w) in zip(synth.SCALE_KEYS, synth.pyramid_shapes(cfgs[f].sphere_W, cfgs[f].sphere_H))}
        rend[f] = mk_renderer(cfgs[f])                           # one renderer per frame: its packed pyramid stays resident
    per = (n_frames + world - 1) // world

    def frame_per_gpu():
        packed = torch.zeros((per, n_pix, 4), dtype=torch.float32, device=dev)
        for i, f in enumerate(mine):
            o = rend[f].render_rays_batch(K, Ts[f], x_rgbs[f], sampled_pixels=pix[f], outputs="minimal")
            packed[i] = sdist.pack_result(o["depth"], o["color"], n_pix)
        if world > 1:
            full = torch.empty((world * per, n_pix, 4), dtype=torch.float32, device=dev)
            dist.all_gather_into_tensor(full, packed)
            return full
        return packed

    def ray_sharded():
        start, stop, pr = sdist.shard_range(n_pix, rank, world)
        packed = torch.zeros((n_frames, pr, 4), dtype=torch.float32, device=dev)
        for f in range(n_frames):
            o = rend[f].render_rays_batch(K, Ts[f], x_rgbs[f], sampled_pixels=pix[f][start:stop], outputs="minimal", ray_offset=start)
            packed[f] = sdist.pack_result(o["depth"], o["color"], pr)
        full = torch.empty((world, n_frames, pr, 4), dtype=torch.float32, device=dev)
        dist.all_gather_into_tensor(full, packed)
        return full

    res = {"workload": "D: 8 frames x 16384 integer pixels x 64 samples, 8 pyramids (1500x452 sphere grid), precision " + args.precision,
           "rays_per_step": n_frames * n_pix, "steps": 3, "warmup": 2}
    ms = max_over_ranks(time_loop(frame_per_gpu, 3, 2, sync), dev, world)
    res["frame_per_gpu"] = {"ms_per_step": ms, "value": n_frames * n_pix / (ms * 1e-3), "unit": "rays/s"}
    if world > 1:
        ms2 = max_over_ranks(time_loop(ray_sharded, 3, 2, sync), dev, world)
        res["ray_sharded"] = {"ms_per_step": ms2, "value": n_frames * n_pix / (ms2 * 1e-3), "unit": "rays/s",
                              "note": "packed pyramids replicated on every rank (resident, like the weights); their one-time broadcast is not in the step"}
        # the two layouts must agree on the frames themselves (Philox noise keyed on (seed, ray index) -> bit-equal)
        for f in need:
            rend[f].seed = 777
        a = frame_per_gpu()
        a = torch.stack([a[(f % world) * per + f // world] for f in range(n_frames)])     # gathered rank-major -> frame order
        for f in need:
            rend[f].seed = 777
        b = ray_sharded().permute(1, 0, 2, 3).reshape(n_frames, -1, 4)[:, :n_pix]
        res["layouts_bit_equal"] = bool(torch.equal(a, b))
        best = "ray_sharded" if ms2 < ms else "frame_per_gpu"
    else:
        best = "frame_per_gpu"
    res["headline_layout"] = best
    res["value"] = res[best]["value"]
    res["unit"] = "rays/s"
    res["tflops_algorithmic"] = res["value"] * flop_per_ray(cfgs[0]) / 1e12
    # keep renderer 0 / pyramid 0 for the lattice query (same class, same sphere grid)
    return res, rend[need[0]], x_rgbs[need[0]], cfgs[need[0]]


def measure_workload_E(args, rank, world, dev, sync, r, x_rgb, cfg):
    """BASELINE.json configs[4] (SURVEY 8d config E): density query of the 256^3 lattice, z-slab per GPU + all-gather."""
    import torch
    from scenerf_b200 import lattice
    K = torch.from_numpy(cfg.K).to(dev)
    ms = max_over_ranks(time_loop(lambda: lattice.density_lattice(r, x_rgb, K, rank=rank, world=world), 3, 1, sync), dev, world)
    n_pts = 256 ** 3
    return {"workload": "E: density query of the 256^3 lattice (16.78 M points), z-slab per GPU + all-gather of the densities, precision " + args.precision,
            "ms_per_step": ms, "value": n_pts / (ms * 1e-3), "unit": "points/s", "steps": 3, "warmup": 1, "scaling": "strong",
            "tflops_algorithmic": n_pts * FLOP_MAIN / (ms * 1e-3) / 1e12, "gpu_launches": int(r.last_lattice_launches)}


def run_render(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from scenerf_b200 import synth
    from scenerf_b200 import dist as sdist
    from scenerf_b200.renderer import B200Renderer

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg, pix_np, desc = workload(args.workload)
    cfg0_tz = cfg.tz
    cfg.tz = cfg.tz + 0.5 * rank                      # frame-per-GPU: every rank renders its own pose of the same source frame
    if args.rays > 0:
        sel = np.random.default_rng(3).permutation(pix_np.shape[0])[:args.rays]
        pix_np = np.ascontiguousarray(pix_np[np.sort(sel)])
        desc += " [diagnostic subset: %d rays]" % pix_np.shape[0]
    R = pix_np.shape[0]
    pm, pg = synth.make_model_params(cfg)
    to_t = lambda d: {k: torch.from_numpy(v) for k, v in d.items()}

    def mk_renderer(c, precision=None, **kw):
        return B200Renderer(hp_from_cfg(c), to_t(pm), to_t(pg), device=dev, precision=precision or args.precision, rng="philox", **kw)

    r = mk_renderer(cfg, skip_zero_chunks=bool(args.skip_zero_chunks), preproject=bool(args.latent_table))
    gen = torch.Generator(device=dev)
    gen.manual_seed(5)                                 # the same source-frame features on every rank (novel poses differ)
    x_rgb = {k: torch.randn((c, h, w), generator=gen, device=dev) * 0.5
             for k, (c, h, w) in zip(synth.SCALE_KEYS, synth.pyramid_shapes(cfg.sphere_W, cfg.sphere_H))}
    K, T = torch.from_numpy(cfg.K), torch.from_numpy(cfg.T)
    pix_host = torch.from_numpy(pix_np).pin_memory()
    pix_dev = pix_host.to(dev)
    r.set_profiling(True)
    outputs = "all" if args.outputs == "all" else "minimal"

    def step_device():
        out = r.render_rays_batch(K, T, x_rgb, sampled_pixels=pix_dev, outputs=outputs)
        if world > 1:
            return sdist.gather_frames(out["depth"], out["color"])
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # `last` holds one step's outputs while the next step allocates its own, in the warm-up as in the timed loop, so that
    # the timed steps reuse cached allocations
    for _ in range(args.warmup):
        last = step_device()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    mlp_ms = []
    launches = 0
    ev0.record()
    for _ in range(args.steps):
        last = step_device()
        launches += r.last_launches
        mlp_ms.append(r.last_mlp_ms()[1])            # waits for this step's main-MLP end event only
    ev1.record()
    barrier()
    clocks = sampler.stop()
    ms_per_step = max_over_ranks(ev0.elapsed_time(ev1), dev, world) / args.steps
    value = world * R / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:
        # one GPU: the dict render_rays_batch returns; N GPUs: the gathered (N, R, 4) [depth, r, g, b] frames
        dump_outputs(args.dump_outputs, last if world == 1 else {"frames": last}, ray_axis=0 if world == 1 else 1)
    del last

    # ---- e2e: host buffers in, host buffers out, through the reference-facing call ------------------------------
    out_host = {"depth": torch.empty((R,), dtype=torch.float32).pin_memory(),
                "color": torch.empty((R, 3), dtype=torch.float32).pin_memory()}

    def step_e2e():
        r.render_rays_batch_host(K, T, x_rgb, pix_host, out_host)
        if world > 1:
            sdist.gather_frames(out_host["depth"].to(dev, non_blocking=True), out_host["color"].to(dev, non_blocking=True))

    e_steps = args.steps if args.e2e_steps <= 0 else args.e2e_steps
    e2e_ms = max_over_ranks(time_loop(step_e2e, e_steps, 1, barrier), dev, world)
    e2e_value = world * R / (e2e_ms * 1e-3)

    # ---- extras every rank takes part in: strong scaling of ONE frame, workload D (both layouts), workload E ----------
    extras = {}
    if not args.no_extras:
        try:
            if world > 1:
                T0 = torch.from_numpy(synth.yaw_translate(cfg.yaw_deg, cfg0_tz))

                def strong():
                    return sdist.render_frame_sharded(
                        lambda p_, off: (lambda o: (o["depth"], o["color"]))(r.render_rays_batch(K, T0, x_rgb, sampled_pixels=p_, outputs="minimal", ray_offset=off)),
                        pix_dev)
                sms = max_over_ranks(time_loop(strong, 3, 1, barrier), dev, world)
                extras["strong"] = {"what": "ONE frame of the workload ray-sharded over %d GPUs (scenerf_b200.dist.render_frame_sharded: contiguous "
                                            "ray ranges + one all-gather of depth+rgb), every rank ends with the full frame" % world,
                                    "ms_per_frame": sms, "value": R / (sms * 1e-3), "unit": "rays/s", "scaling": "strong", "steps": 3, "warmup": 1,
                                    "one_gpu_ms_per_frame": ms_per_step, "speedup": ms_per_step / sms, "efficiency": ms_per_step / sms / world,
                                    "note": "one_gpu_ms_per_frame = this run's frame-per-GPU step (same work per GPU as a 1-GPU frame, plus the gather)"}
            d_res, rD, xD, cD = measure_workload_D(args, rank, world, dev, barrier, mk_renderer)
            extras["workload_D"] = d_res
            extras["workload_E"] = measure_workload_E(args, rank, world, dev, barrier, rD, xD, cD)
            del rD, xD
        except Exception as e:                      # extras are informational; never lose the headline line
            extras["error"] = "%s: %s" % (type(e).__name__, str(e).splitlines()[0] if str(e) else "")
        torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (main point-MLP pass), measured live with CUDA events ------------------
    peaks = load_peaks()
    peak = peaks.get("bf16_tflops_sustained") or 1400.0
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (fp16 and bf16 share the tcgen05 kind::f16 rate; the kernel runs inside a seconds-long step)" \
        if peaks else "fallback 1.4 PF sustained (B200_PROFILING.md)"
    main_ms = float(np.mean([m for m in mlp_ms if m > 0])) if mlp_ms else float("nan")
    flop_launch = float(R) * cfg.S * FLOP_MAIN
    achieved = flop_launch / (main_ms * 1e-3) / 1e12
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(args.workload + "_" + args.precision)
    except Exception:
        pass
    mma_mult = 4.0 if args.precision == "fp32tc" else 1.0
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_unit": "DRAM bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum, profiles/traffic.json)",
                "kernel": "point_mlp_tc_kernel (main pass)" if args.precision != "fp32" else "sgemm_nt_kernel chain",
                "kernel_ms": main_ms, "algorithmic_flop_per_launch": flop_launch, "peak_source": peak_src,
                "executed_tensor_tflops": achieved * mma_mult * 1.025, "executed_frac": achieved * mma_mult * 1.025 / peak,
                "peak_burst": peaks.get("bf16_tflops"), "executed_frac_of_burst": (achieved * mma_mult * 1.025 / peaks["bf16_tflops"]) if peaks.get("bf16_tflops") else None,
                "note": "achieved = ALGORITHMIC flops (10 811 392 per sample point) / kernel time, per GPU (rank 0's launch). " +
                        ("fp32tc issues 4 fp16 MMAs per algorithmic product, (x_hi,x_lo) x (W_hi,W_lo): executed_* = 4 x 1.025 (K/N padding) x algorithmic, "
                         "i.e. frac can reach 0.25 of the kind::f16 rate at most; executed_frac is the tensor-pipe figure.  It can exceed 1 against the "
                         "SUSTAINED peak: cuBLAS sustains 1456 TFLOP/s at ~1.4 GHz under the 1 kW cap while this kernel holds ~1.65 GHz "
                         "(clocks in this line); executed_frac_of_burst is against the 1709 TFLOP/s burst figure" if args.precision == "fp32tc"
                         else "executed = 1.025 x algorithmic (K padded 42->64, 2480->2496, N 4->16)"),
                "whole_step_tflops_per_gpu": R * flop_per_ray(cfg) / (ms_per_step * 1e-3) / 1e12}

    # ---- variants measured in the same run (not the headline) --------------------------------------------------------
    variants = {}

    def quick(rr, n=None, steps=3, warm=2, outs="minimal"):
        p_ = pix_dev if n is None else pix_dev[:n]
        ms_ = time_loop(lambda: rr.render_rays_batch(K, T, x_rgb, sampled_pixels=p_, outputs=outs), steps, warm, torch.cuda.synchronize)
        return {"ms_per_step": ms_, "value": p_.shape[0] / (ms_ * 1e-3), "unit": "rays/s"}

    try:
        if args.no_variants:
            raise RuntimeError("variants disabled (--no-variants)")
        if args.precision != "fp16":
            rf = mk_renderer(cfg, "fp16")
            rf.set_profiling(True)
            v = quick(rf)
            fm = rf.last_mlp_ms()[1]
            v.update({"precision": PREC_DESC["fp16"], "kernel_ms": fm, "roofline_frac": flop_launch / (fm * 1e-3) / 1e12 / peak,
                      "note": "round-1 headline mode; parity tolerance depth <= 3e-4*max_depth, colour <= 1e-3 (tests/test_gpu_parity.py)"})
            variants["fast"] = v
            del rf
        rs = mk_renderer(cfg, skip_zero_chunks=not bool(args.skip_zero_chunks))
        v = quick(rs)
        v["note"] = "lin_z K-chunks whose gathered features are zero for the whole tile pair are skipped; results bit-identical; algorithmic rays/s"
        variants["skip_zero_chunks=%s" % (not bool(args.skip_zero_chunks))] = v
        del rs
        if outputs == "minimal":
            v = quick(r, outs="all")
            v["note"] = "the reference's full 12-key dict incl. RaySOM (scenerf.py:456-469): +%d B/ray of output writes" % ((19 + 4 * cfg.S) * 4 - 16)
            variants["outputs=all"] = v
        # pre-projected latent table (exact restructuring, SURVEY 7 hard part 3b): lin_z of the main network tabulated per
        # sphere pixel once per image, 70.5 % of the per-point FLOPs never executed.  EXECUTED flops are reported apart
        # from the algorithmic ones and never enter the roofline line above.
        def table_variant(prec):
            rp = mk_renderer(cfg, prec, preproject=True)
            rp.set_profiling(True)
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            rp.render_rays_batch(K, T, x_rgb, sampled_pixels=pix_dev[:256], outputs="minimal")
            t1.record()
            torch.cuda.synchronize()
            v_ = quick(rp)
            km = rp.last_mlp_ms()[1]
            ems_ = time_loop(lambda: rp.render_rays_batch_host(K, T, x_rgb, pix_host, out_host), 3, 1, torch.cuda.synchronize)
            exec_flop = float(R) * cfg.S * 2 * 1596416.0          # lin_in + 6 x 512x512 + lin_out per point
            v_.update({"precision": prec, "kernel_ms": km, "e2e": {"value": R / (ems_ * 1e-3), "unit": "rays/s", "ms_per_frame": ems_},
                       "first_call_ms_incl_pack_and_table": t0.elapsed_time(t1),
                       "table_mb": rp._tab_buf.numel() / 1e6, "table_build_launches": rp.last_pack_launches,
                       "executed_tflops": exec_flop / (km * 1e-3) / 1e12 * (4.0 if prec == "fp32tc" else 1.0),
                       "algorithmic_tflops": flop_launch / (km * 1e-3) / 1e12,
                       "note": "lin_z[b](z) of the main network read from a per-sphere-pixel table built once per image (srf_build_latent_table); "
                               "executed MMA flops = 3.19 MFLOP/point (x4 issued in fp32tc) vs 10.81 algorithmic; value is ALGORITHMIC rays/s"})
            del rp
            torch.cuda.empty_cache()
            return v_
        if args.precision != "fp32" and not args.no_table_variant:
            variants["latent_table (%s)" % args.precision] = table_variant(args.precision)
            if args.precision != "fp16":
                variants["latent_table (fp16)"] = table_variant("fp16")
        if args.precision != "fp32":
            n32 = min(R, 16384)
            r32 = mk_renderer(cfg, "fp32")
            v = quick(r32, n=n32, steps=1, warm=1)
            v["sample"] = "%d rays" % n32
            variants["precision=fp32 (strict SIMT mode)"] = v
            del r32
    except Exception as e:          # variants are informational; never lose the headline line
        variants["error"] = str(e).splitlines()[0]

    cpu = None
    parity = None
    if not args.no_cpu_baseline:
        pyr_cpu = {k: v.detach().cpu().numpy() for k, v in x_rgb.items()}
        if world == 1:
            cpu = cpu_baseline(args.workload, cfg, pix_np, pyr_cpu)
        # parity of this very run: same rays, weights, pyramid and noise through the oracle and through the GPU path
        from oracle.scenerf_oracle import OracleRenderer
        n = 64
        rng = np.random.default_rng(1)
        sel = rng.permutation(R)[:n]
        nu = rng.random((n, cfg.n_pts_uni), dtype=np.float32)
        nn_ = rng.standard_normal((n, cfg.n_gaussians * cfg.n_pts_per_gaussian)).astype(np.float32)
        ref = OracleRenderer(cfg, pm, pg).render_rays_batch(cfg.K, cfg.T, pyr_cpu, pix_np[sel], n, nu, nn_)
        got = r.render_rays_batch(K, T, x_rgb, sampled_pixels=torch.from_numpy(pix_np[sel]), outputs="minimal",
                                  noise=(torch.from_numpy(nu), torch.from_numpy(nn_)))
        parity = {"rays": n, "depth_max_abs_err_m": float(np.abs(got["depth"].cpu().numpy() - ref["depth"]).max()),
                  "color_max_abs_err": float(np.abs(got["color"].cpu().numpy() - ref["color"]).max()),
                  "vs": "CPU oracle (pinned to the reference at this very size by tests/golden/full_*.npz), identical rays/weights/noise",
                  "tolerance": "depth <= 2e-4*max_sample_depth, colour <= 2e-4 (fp32 / fp32tc); depth <= 3e-4*max_sample_depth, colour <= 1e-3 (fp16)"}

    fmt = "fp16" if args.precision == "fp16" else "fp32"
    pyr_mb = sum(c * h * w for c, h, w in synth.pyramid_shapes(cfg.sphere_W, cfg.sphere_H)) * (2 if fmt == "fp16" else 4) / 1e6
    line = {"metric": "rays/sec", "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": PREC_DTYPE[args.precision], "data": "synthetic",
            "config": {"workload": desc, "rays_per_gpu": R, "samples_per_ray": cfg.S, "parallelism": "frame-per-GPU x%d (one pose of the source frame per GPU + all-gather of depth+rgb)" % world,
                       "precision": args.precision + ": " + PREC_DESC[args.precision],
                       "skip_zero_chunks": bool(args.skip_zero_chunks), "latent_table": bool(args.latent_table), "outputs": "depth+color" if outputs == "minimal" else "the reference's 12-key dict",
                       "l2": "inputs larger than L2: %.0f MB %s pyramid + %d MB weights + 1.9 GB of per-step intermediates (points, raw MLP output); no flush needed"
                             % (pyr_mb, fmt, 44 if args.precision == "fp32tc" else 22)},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": R * 2 * 4, "d2h_bytes_per_step": R * 4 * 4, "steps": e_steps},
            "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu, "parity": parity, "variants": variants}
    line.update(extras)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="B", choices=["A", "B", "Bp", "C", "D", "E", "sweep", "train", "decoder"])
    ap.add_argument("--train-matmul", default="fp32", choices=["fp32", "tf32"], help="--workload train: GEMM engine")
    ap.add_argument("--sweep-poses", type=int, default=63)
    ap.add_argument("--sweep-scale", type=int, default=2)
    ap.add_argument("--sweep-table", type=int, default=1, help="--workload sweep: 1 = use the per-image latent table (default), 0 = dense")
    ap.add_argument("--precision", default="fp32tc", choices=["fp32tc", "fp16", "fp32"],
                    help="fp32tc (default, precision-matched to the reference's fp32 sgemm), fp16 (fast mode), fp32 (strict SIMT)")
    ap.add_argument("--outputs", default="minimal", choices=["minimal", "all"], help="depth+colour (inference callers) or the full 12-key dict")
    ap.add_argument("--skip-zero-chunks", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--rays", type=int, default=0, help="diagnostics: use only the first N rays of the workload")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--no-table-variant", action="store_true")
    ap.add_argument("--latent-table", type=int, default=0, help="1: the timed renderer uses the pre-projected latent table (diagnostics / profiling)")
    ap.add_argument("--no-extras", action="store_true", help="skip the strong-scaling / workload D / workload E measurements")
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps of the host-buffer (e2e) loop; 0 = same as --steps")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last timed step as DIR/<name>.npy (float32, at most "
                         "64 MB in all: a fixed, seeded sample of rays beyond that); render workloads A, B, Bp and C")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload not in ("A", "B", "Bp", "C")):
        ap.error("--dump-outputs applies to --impl ours with the render workloads A, B, Bp and C")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if args.workload in ("D", "E", "sweep", "train", "decoder"):
            args.workload = "B"
        run_reference(args, rank, world)
        return
    if args.workload == "sweep":
        run_sweep(args, rank, world, local_rank)
        return
    if args.workload == "train":
        run_train(args, rank, world, local_rank)
        return
    if args.workload == "E":
        run_lattice(args, rank, world, local_rank)
        return
    if args.workload == "D":
        run_D(args, rank, world, local_rank)
        return
    if args.workload == "decoder":
        run_decoder(args, rank, world, local_rank)
        return
    run_render(args, rank, world, local_rank)


def run_decoder(args, rank, world, local_rank):
    """--workload decoder: the producer tail (SURVEY 8f-3).  One step = DecoderSphere.forward of ONE KITTI image at the reference's
    real sizes (EfficientNet-B7 maps of a 1220x370 image, num_features = bottleneck = 2560, sphere grid 1500x452) through
    scenerf_b200.decoder.SphereDecoderB200: conv2 (PyTorch), 6 sphere resamplings, 5 x (upsample+concat, 7 implicit-GEMM convolutions),
    the last convolution of each level writing the packed fp32 + fp16 pyramid.  Synthetic weights, maps and pixel->sphere table."""
    import torch
    from scenerf_b200 import synth
    from scenerf_b200.decoder import SphereDecoderB200
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    W, H, oW, oH, F = 1220, 370, 1500, 452, 2560
    gen = torch.Generator(device=dev)
    gen.manual_seed(3)
    rnd = lambda *sh: torch.randn(sh, generator=gen, device=dev)
    state = {}
    state["conv2.weight"] = rnd(F, F, 1, 1) * (2.0 / F) ** 0.5
    state["conv2.bias"] = rnd(F) * 0.1
    flop = 0.0
    dims = {s: (round(oH / s), round(oW / s)) for s in (1, 2, 4, 8, 16)}
    for s, (cin, cout) in synth.decoder_level_channels(F).items():
        pre = "up%d._net." % s
        px = dims[s][0] * dims[s][1]
        state[pre + "0.weight"] = rnd(cout, cin, 3, 3) * (2.0 / (9 * cin)) ** 0.5
        state[pre + "0.bias"] = rnd(cout) * 0.1
        flop += 2.0 * 9 * cin * cout * px
        for blk in (1, 2, 3):
            for cb in (1, 2):
                n = pre + "%d.conv_block%d" % (blk, cb)
                state[n + ".0.weight"] = rnd(cout, cout, 3, 3) * (2.0 / (9 * cout)) ** 0.5
                state[n + ".0.bias"] = rnd(cout) * 0.1
                state[n + ".1.weight"] = 1.0 + 0.1 * rnd(cout)
                state[n + ".1.bias"] = 0.1 * rnd(cout)
                state[n + ".1.running_mean"] = 0.1 * rnd(cout)
                state[n + ".1.running_var"] = 1.0 + 0.2 * torch.rand(cout, generator=gen, device=dev)
                flop += 2.0 * 9 * cout * cout * px
    dec = SphereDecoderB200(state, oW, oH, device=dev, emit_fp16=True)
    del state
    chans = {1: 3, 2: 32, 4: 48, 8: 80, 16: 224, 32: F}
    features = [None] * 12
    for idx, sc in ((0, 1), (4, 2), (5, 4), (6, 8), (8, 16), (11, 32)):
        features[idx] = rnd(1, chans[sc], -(-H // sc), -(-W // sc))
    ys, xs = torch.meshgrid(torch.arange(H, device=dev), torch.arange(W, device=dev), indexing="ij")
    pix = torch.stack([xs.reshape(-1), ys.reshape(-1)], 1).float()
    pix_sphere = torch.stack([torch.round(pix[:, 0] * ((oW - 1) / (W - 1))), torch.round(pix[:, 1] * ((oH - 1) / (H - 1)))], 1).long()
    ms = time_loop(lambda: dec(features, pix, pix_sphere), args.steps, args.warmup, torch.cuda.synchronize)
    peaks = load_peaks()
    peak = float(peaks.get("bf16_tflops_sustained") or 1400.0) / 2.0
    if rank == 0:
        print(json.dumps({"metric": "decoder images/sec (DecoderSphere.forward of one 1220x370 KITTI image -> packed 1500x452 pyramid)",
                          "value": 1e3 / ms, "unit": "images/s", "ms_per_step": ms, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
                          "dtype": "tf32 operands (rounded to nearest), fp32 storage and accumulate", "data": "synthetic", "higher_is_better": True,
                          "gpu_launches": int(dec.launches) + 18,
                          "roofline": {"bound": "tensor (tcgen05 kind::tf32; peak = measured bf16 sustained / 2)", "achieved": flop / (ms * 1e-3) / 1e12,
                                       "peak": peak, "unit": "TFLOP/s", "frac": flop / (ms * 1e-3) / 1e12 / peak,
                                       "algorithmic_flop_per_step": flop,
                                       "note": "whole step incl. conv2 (PyTorch), the sphere resamplings and the upsample+concat kernels; "
                                               "algorithmic flops = 2*9*Cin*Cout per output pixel of the 35 convolutions"}}))


def run_D(args, rank, world, local_rank):
    """--workload D standalone: the same measurement as the `workload_D` object of the default line."""
    import torch
    import torch.distributed as dist
    from scenerf_b200 import synth
    from scenerf_b200.renderer import B200Renderer
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    pm, pg = synth.make_model_params(synth.config_A())
    to_t = lambda d: {k: torch.from_numpy(v) for k, v in d.items()}
    mk = lambda c: B200Renderer(hp_from_cfg(c), to_t(pm), to_t(pg), device=dev, precision=args.precision, rng="philox")

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    res, _, _, _ = measure_workload_D(args, rank, world, dev, sync, mk)
    if rank == 0:
        res.update({"metric": "rays/sec", "n_gpus": world, "higher_is_better": True, "dtype": PREC_DTYPE[args.precision], "data": "synthetic",
                    "scaling": "strong"})
        print(json.dumps(res))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
