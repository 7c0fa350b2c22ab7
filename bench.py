#!/usr/bin/env python
"""Benchmark of the ray-march hot path (BASELINE.json metric: rays/sec, 512x512, 128 samples/ray,
3 source views, 18 keypoints).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config {2,3,4,5}] [--scene {ones,hull}] [--impl reference]
                    [--dump-outputs DIR]

A step = one pass of the hot path over one synthetic frame: re-layout of the (new) source feature
maps + ray generation + sampling + shading + compositing for every pixel of the novel view.

BASELINE.json configs (config 1 is the reference's CPU-runnable plumbing case: a parity test, not a bench line):
  2 (default, the headline)  512x512, 128 samples/ray.  N > 1 ranks: one novel view per rank (= config 5, weak scaling).
  3                          512x512, 64 coarse + 64 fine samples, early-ray termination at 1e-4; ranks as in 2.
  4                          ONE 1024x1024 frame, 128 samples/ray, split into lattice phases over the N ranks (strong scaling).
  5                          alias of 2 (the render_dynamic.py-style sweep: one 512x512 view per GPU).
The frames are exchanged with ONE NCCL all-gather.

`value`   : inputs resident in HBM, CUDA-event time on the launch stream, max over ranks.
`e2e`     : the same metric through the reference-facing API (`KeypointNeRF.render_pifu_nerf`) with
            pinned HOST tensors in and host tensors out (H2D + D2H inside the timed region).
`roofline`: the dominant kernel (shade_geo_vseq_kernel at 18 keypoints, shade_geo_kernel at 24): algorithmic FLOPs of the samples it shaded / its device time, both
            measured live (valid-sample counter of the launch, CUDA events around the kernel on the launch stream inside the
            timed region), against the measured dense bf16 tensor peak in MEASURED_PEAKS.json; `pair` adds the colour kernel
            (executed FLOPs: 419 200 per valid sample + 79 536 per sample with density > 0).
`--dump-outputs DIR`: after the timed steps, rank 0 writes what the render of the last timed step returned (every output plane
            of its frame, and with N > 1 ranks the all-gathered frames) as DIR/<name>.npy in float32; should that exceed 64 MB, every
            array keeps the same fixed, seeded sample of its pixels (the last two axes flattened).  The inputs are generated from
            fixed seeds, so two builds run with the same arguments can be compared output for output.
`cpu_baseline` / `--impl reference`: the CPU oracle port (oracle/, torch-CPU, all host threads) on a bounded sample of the
            same workload (a strided pass of the same frame: 4096 rays, fewer when that would take too long).
"""
from __future__ import annotations

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

N_KPT = 18
N_VIEWS = 3
CONFIGS = {
    2: dict(size=512, S_c=128, S_f=0, fine=False, ert=0.0, part="views",
            workload="512x512 frame, 128 samples/ray (fine off), 3 source views 512^2, 18 keypoints, random maps+weights"),
    3: dict(size=512, S_c=64, S_f=64, fine=True, ert=1e-4, part="views",
            workload="512x512 frame, 64 coarse + 64 fine samples/ray, early-ray termination 1e-4, 3 source views 512^2, "
                     "18 keypoints, random maps+weights"),
    4: dict(size=1024, S_c=128, S_f=0, fine=False, ert=0.0, part="lattice",
            workload="1024x1024 frame, 128 samples/ray (fine off), 3 source views 512^2, 18 keypoints, random maps+weights"),
}
CONFIGS[5] = CONFIGS[2]


def flops(n_kpt: int, n_views: int):
    """Dense-layer FLOPs (2*MAC), SURVEY.md section 8a: (per valid sample: geometry MLP of every view + pooled density tail +
    compress layer, per sample with density > 0: the IBR colour head of every view)."""
    enc = 7 * n_kpt
    geo = (enc + 64) * 128 + 128 * 128 + 136 * 120 + 120 * 64
    ibr = 4 * 16 + 16 * 35 + 105 * 64 + 64 * 32 + 32 * 32 + 32 * 33 + 32 * 32 + 32 + 37 * 16 + 16 * 8 + 8
    pooled = 128 * 64 + 64 * 64 + 64 * 2 + 128 * 24
    return 2 * (n_views * geo + pooled), 2 * n_views * ibr


def ncu_traffic():
    """DRAM bytes per launch of the shading kernels from the latest committed ncu capture (profiles/*_traffic.json, written
    by tools/summarize_profile.py); None when no capture is committed."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json")))
    if not files:
        return None, None, None
    d = json.load(open(files[-1]))
    per = {k: v.get("dram__bytes_read.sum", 0.0) + v.get("dram__bytes_write.sum", 0.0) for k, v in d["kernels"].items()}
    geo = next((v for k, v in per.items() if "geo" in k), None)
    return geo, sum(per.values()), os.path.basename(files[-1])


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"tflops": float(d.get("bf16_tflops_sustained", d.get("bf16_tflops"))), "hbm_gbs": float(d["hbm_gbs"]),
                "source": "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)"}
    return {"tflops": 1400.0, "hbm_gbs": 6650.0, "source": "B200_PROFILING.md fallback, sustained (of fallback)"}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def cpu_port_rays_per_s(cfg: dict, scene_kind: str, steps: int, warmup: int, budget_s: float = 150.0):
    """Oracle port on ALL host cores (set explicitly: under torchrun OMP_NUM_THREADS is 1).  One step = the first `rays` pixels of
    a 64x64 strided pass of the configured frame; `rays` starts at 4096 (a full pass) and is cut (to a multiple of 64, at least
    256) when the first untimed pass says `steps` passes would exceed `budget_s`, so that the run ends within a few minutes
    whatever --steps the caller asks for.  The torch-CPU path is bound by materialised intermediates and may run faster on 16
    threads than on every core of a large host: the first two untimed passes try both and the timed ones use the faster."""
    import torch
    from keypointnerf_b200 import synthetic as syn
    from oracle import kpnerf_oracle as O
    scene = syn.make_scene(512, N_VIEWS, N_KPT, fg_mode=scene_kind)
    fw = O.fold_weights(syn.make_weights(N_KPT))
    target = syn.make_target(cfg["size"], azimuth=1.0)
    step = cfg["size"] // 64

    def one_pass(i, rays):
        pix = O.pixel_lattice(cfg["size"], cfg["size"], step, i % step, (i // step) % step)[:rays]
        t0 = time.perf_counter()
        O.render_pixels(scene, fw, target, pix, cfg["S_c"], cfg["S_f"], cfg["fine"])
        return time.perf_counter() - t0

    with torch.no_grad():
        all_cores = os.cpu_count() or 1
        torch.set_num_threads(all_cores)
        rays = 4096
        one_pass(0, 256)                         # first call of the process: allocator / thread-pool warm-up, not a measurement
        probe = {}
        for n in sorted({all_cores, min(16, all_cores)}, reverse=True):
            torch.set_num_threads(n)
            probe[n] = one_pass(1, 1024)
        torch.set_num_threads(min(probe, key=probe.get))
        cores = torch.get_num_threads()
        est = min(probe.values()) * 4.0 * (steps + warmup)
        if est > budget_s:
            rays = max(256, int(4096 * budget_s / est) // 64 * 64)
        times = []
        for i in range(warmup + steps):
            dt = one_pass(i, rays)
            if i >= warmup:
                times.append(dt)
    return rays * len(times) / sum(times), cores, sum(times) / len(times) * 1e3, rays


def run_reference_arm(args, cfg, out_fd):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    val, cores, ms, rays = cpu_port_rays_per_s(cfg, args.scene, args.steps, args.warmup)
    sample = (f"the first {rays} rays of a 64x64 strided pass of the frame per step ({rays} rays x {cfg['S_c'] + cfg['S_f']} "
              f"samples), {cores} threads")
    line = {"impl": "reference", "metric": "rays/sec", "value": val, "unit": "rays/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong" if cfg["part"] == "lattice" else "weak",
            "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": {"workload": cfg["workload"], "note": "CPU oracle port of the reference PyTorch path (the reference is "
                       "Python and cannot travel to the GPU box); bounded sample per step"},
            "cpu_baseline": {"value": val, "unit": "rays/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    _emit(out_fd, line)
    return 0


def _private_stdout():
    """The contract is ONE JSON line on stdout: libraries (NCCL prints its version banner there) get stderr instead."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return saved


def _emit(fd: int, line: dict):
    os.write(fd, (json.dumps(line) + "\n").encode())


def main():
    out_fd = _private_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--scene", default="ones", choices=["ones", "hull"],
                    help="ones: SURVEY.md 8d recipe (all-foreground masks, ~46 %% of the samples valid); hull: silhouette masks "
                         "(~1.6 %% valid, like real captures)")
    ap.add_argument("--engine", type=int, default=0)
    ap.add_argument("--n-kpt", type=int, default=N_KPT)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-steps", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        return run_reference_arm(args, cfg, out_fd)
    if args.warmup < 3:
        args.warmup = 3

    import numpy as np
    import torch
    import torch.distributed as dist

    import __graft_entry__ as G
    from keypointnerf_b200 import distributed as D
    from keypointnerf_b200 import synthetic as syn
    from keypointnerf_b200.testing import build_model, scene_tensors

    G.build()
    rank, world, local = D.init_from_env("nccl")
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torchrun for N>1)"
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    size, S_c, S_f, fine, ert = cfg["size"], cfg["S_c"], cfg["S_f"], cfg["fine"], cfg["ert"]
    lattice = cfg["part"] == "lattice"
    n_kpt = args.n_kpt

    scene = syn.make_scene(512, N_VIEWS, n_kpt, fg_mode=args.scene)
    weights = syn.make_weights(n_kpt)
    # config 4: every rank renders its lattice phase of the SAME view; otherwise one novel view per rank
    target = syn.make_target(size, azimuth=1.0 if lattice else 1.0 + rank * np.pi / 4.0)
    net = build_model(weights, n_kpt, dev)
    net.engine = args.engine
    a = scene_tensors(scene, target, dev)
    h = scene_tensors(scene, target, "cpu", pin=True)
    m = net.marcher()
    m.reserve(size * size // (world if lattice else 1), S_c + S_f)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    kw = dict(S_c=S_c, S_f=S_f, fine=fine, engine=args.engine, ert_eps=ert)
    key = "tex_fg_fine" if fine else "tex_fg"
    gev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    gstate = {"k": -1}

    def bind(t):
        m.set_scene(KRT=t["cam"]["KRT"], extrin=t["sp_data"]["extrin"], kpt3d=t["sp_data"]["kpt3d"].reshape(-1, 3),
                    bounds=t["bounds"], feat64=t["feat_geo"][0], feat8=t["feat_geo"][1], feat_tex=t["feat_tex"],
                    img=t["img"], fg=t["fg"], width=scene["width"], height=scene["height"], znear=scene["znear"],
                    zfar=scene["zfar"], nml_scale=scene["nml_scale"])

    def step_device():
        bind(a)   # every step is a new frame: the atlases are re-packed
        k = gstate["k"]
        if lattice:
            y0, x0, sy, sx = D.lattice_phase(rank, world)
            res = m.render(K=a["cam_tar"]["K"], RT=a["cam_tar"]["RT"], znear=target["znear"], zfar=target["zfar"], x0=x0, y0=y0,
                           step=sx, step_y=sy, nx=size // sx, ny=size // sy, out_device="cuda", **kw)
            if k >= 0:
                gev[k][0].record()
            out = D.gather_lattice(res[key], world)
        else:
            res = m.render(K=a["cam_tar"]["K"], RT=a["cam_tar"]["RT"], znear=target["znear"], zfar=target["zfar"],
                           x0=0, y0=0, step=1, nx=size, ny=size, out_device="cuda", **kw)
            if k >= 0:
                gev[k][0].record()
            out = D.gather_views(res[key], world)
        if k >= 0:
            gev[k][1].record()
        if k == args.steps - 1:
            gstate["res"], gstate["out"] = res, out   # what --dump-outputs writes
        return out

    cfgk = dict(sample_per_ray_c=S_c, sample_per_ray_f=S_f, fine=fine, uniform=True, ert_eps=ert)
    level = int(np.log2(size)) - 5   # render_novel_views: max(0, log2(im_h) - 5), reference src/model.py:485

    def step_e2e():
        net._scene_key = None   # new frame: host feature maps are uploaded again
        return net.render_pifu_nerf(net, h["img"], h["cam"], h["cam_tar"], level=level, sp_data=h["sp_data"],
                                    feat_geo=h["feat_geo"], feat_tex=h["feat_tex"], src_foreground_mask=h["fg"],
                                    bounds=h["bounds"], mask_at_box=None, dist_shard=(rank, world) if lattice else None, **cfgk)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    import gc
    gc.collect()
    gc.disable()   # no collector pauses inside the timed loops (timeit does the same); re-enabled below
    for _ in range(args.warmup):
        step_device()
    barrier()
    m.stats()           # drain event pool / counters
    launches0 = m.stats()["kernel_launches"]
    m.set_profiling(True)
    sampler = ClockSampler(local)
    sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    t_wall0 = time.perf_counter()
    for k in range(args.steps):
        flush.zero_()                      # L2 flush between timed iterations (not timed)
        gstate["k"] = k
        evs[k][0].record()
        step_device()
        evs[k][1].record()
    gstate["k"] = -1
    barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop()
    st = m.stats()   # counters of the LAST step's render, event times summed over the timed steps
    m.set_profiling(False)
    if args.dump_outputs and rank == 0:
        dump = dict(gstate["res"])
        if world > 1:
            dump["gathered_" + key] = gstate["out"]
        limit, total = 64 << 20, sum(v.numel() * 4 for v in dump.values())
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, v in dump.items():
            a = v.float().cpu().numpy()
            if total > limit:
                a = a.reshape(*a.shape[:-2], -1)
                n = a.shape[-1]
                a = a[..., np.sort(np.random.default_rng(0).choice(n, n * limit // total, replace=False))]
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    ms_rank = sum(e0.elapsed_time(e1) for e0, e1 in evs)
    gather_ms = sum(e0.elapsed_time(e1) for e0, e1 in gev)
    mine = torch.tensor([ms_rank, st["shade_ms"], st["geo_ms"], gather_ms, float(st["samples_valid"]), float(st["samples_coloured"])],
                        dtype=torch.float64, device=dev)
    per_rank = D.gather_views(mine, world).cpu().numpy()
    ms_total = float(per_rank[:, 0].max())
    rays_per_step = size * size * (1 if lattice else world)
    value = rays_per_step * args.steps / (ms_total * 1e-3)
    launches = st["kernel_launches"] - launches0

    # end to end through the reference-facing API, host buffers in / host buffers out
    out = None
    for _ in range(3):
        out = step_e2e()      # keep the previous result alive like the timed loop does (two sets of pinned output buffers)
    barrier()
    e2e_each = []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        t1 = time.perf_counter()
        out = step_e2e()      # returns host tensors: the call itself waits for the device-to-host copies
        e2e_each.append((time.perf_counter() - t1) * 1e3)
    barrier()
    te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    gc.enable()
    e2e_val = rays_per_step * args.steps / float(te.item())
    h2d = sum(int(t.numel() * t.element_size()) for t in
              [h["feat_geo"][0], h["feat_geo"][1], h["feat_tex"], h["img"], h["fg"], h["cam"]["KRT"], h["sp_data"]["extrin"],
               h["sp_data"]["kpt3d"], h["bounds"], h["cam_tar"]["K"], h["cam_tar"]["RT"]])
    d2h = sum(int(v.numel() * v.element_size()) for v in out.values())

    f_geo, f_ibr = flops(n_kpt, N_VIEWS)
    pk = peaks()
    n_eval = size * size * (S_c + (S_c + S_f if fine else 0)) // (world if lattice else 1)   # samples evaluated per rank and step
    valid, coloured = st["samples_valid"], st["samples_coloured"]
    geo_ms, shade_ms = st["geo_ms"], st["shade_ms"]
    ach_geo = f_geo * valid * args.steps / (geo_ms * 1e-3) / 1e12 if geo_ms > 0 else None
    ach_pair = (f_geo * valid + f_ibr * coloured) * args.steps / (shade_ms * 1e-3) / 1e12 if shade_ms > 0 else None
    t_geo, t_pair, t_src = ncu_traffic()
    vseq = n_kpt == 18 and args.engine in (0, 3)   # the library's choice of geometry kernel (include/kpnerf_b200.h, kpn_opts.engine)
    gk = "shade_geo_vseq_kernel" if vseq else "shade_geo_kernel"
    roofline = {"bound": "tensor", "kernel": gk + " (gather + keypoint encoding + geometry MLP + pooling + density tail)",
                "achieved": ach_geo, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": (ach_geo / pk["tflops"]) if ach_geo else None,
                "traffic": t_geo, "traffic_unit": "DRAM bytes per launch (one chunk = one 512x512x128 frame), ncu --set full",
                "traffic_source": t_src, "peak_source": pk["source"],
                "flop_per_valid_sample": f_geo, "flop_per_coloured_sample": f_ibr,
                "valid_samples_per_step": valid, "coloured_samples_per_step": coloured,
                "valid_frac": valid / float(n_eval), "geo_ms_per_step": geo_ms / args.steps,
                "pair": {"kernels": gk + " + shade_color_kernel", "achieved": ach_pair,
                         "frac": (ach_pair / pk["tflops"]) if ach_pair else None, "ms_per_step": shade_ms / args.steps,
                         "traffic": t_pair},
                "shade_launches_per_step": st["shade_launches"] / args.steps,
                "shade_share_of_step": (shade_ms / ms_rank) if ms_rank else None,
                "nominal_tflops_all_samples": (f_geo + f_ibr) * n_eval * args.steps / (ms_rank * 1e-3) / 1e12}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        val, cores, ms, rays = cpu_port_rays_per_s(cfg, args.scene, args.cpu_steps, 1)
        cpu = {"value": val, "unit": "rays/s", "cores": cores, "kind": "port",
               "sample": f"{args.cpu_steps} x the first {rays} rays of a 64x64 strided pass of the same frame ({rays} rays x "
                         f"{S_c + S_f} samples), {ms:.0f} ms each, torch-CPU oracle port"}

    if rank == 0:
        part = (f"one {size}x{size} frame in {world} lattice phases (one per GPU), one all-gather of the phases" if lattice else
                f"one novel view per GPU x{world}, one all-gather of frames")
        names = ["ms", "shade_ms", "geo_ms", "all_gather_ms", "valid_samples", "coloured_samples"]
        line = {"metric": "rays/sec", "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
                "scaling": "strong" if lattice else "weak",
                "vs_baseline": None, "dtype": "fp32" if args.engine == 1 else net.marcher_dtype(), "data": "synthetic",
                "config": {"workload": cfg["workload"], "baseline_config": args.config, "parallelism": part,
                           "scene": f"{args.scene} foreground masks", "n_kpt": n_kpt,
                           "l2": "flushed between timed iterations (256 MiB write)", "gc": "python collector off inside the timed loops", "engine": args.engine,
                           "wall_ms_per_step_incl_flush": t_wall / args.steps * 1e3},
                "clocks": clocks,
                "e2e": {"value": e2e_val, "unit": "rays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_each": [round(x, 2) for x in e2e_each]},
                "gpu_launches": launches, "roofline": roofline,
                "per_rank": [{n: (float(v) / args.steps if n.endswith("ms") else float(v)) for n, v in zip(names, row)}
                             for row in per_rank],
                "cpu_baseline": cpu}
        _emit(out_fd, line)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
