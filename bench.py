#!/usr/bin/env python
"""Benchmark of the NeuMesh rendering hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the reference algorithm's CPU path (oracle port)

One step = one 800x800 frame of the synthetic spiral (640 000 rays, the configuration BASELINE.json's metric is quoted
on: icosphere mesh V = 163 842, 32-d vertex codes, K = 8, calc_normal + white background, bounded near/far, 64 + 64
samples).  Prints ONE JSON line (rank 0).  Keys are documented in DESIGN.md "Measurement".
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

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from neumesh_b200 import synth  # noqa: E402

H = W = 800
MESH_LEVEL = 7
RENDER_KW = dict(calc_normal=True, white_bkgd=True, bounded_near_far=True)
METRIC = "rays_per_sec_800x800_spiral"
DEFAULT_ENGINE = "tcgen05_f16"
CODE_DIM = 32
WORKLOAD_NAME = "spiral_800x800_icosphere_V163842_F32_K8"

# BASELINE.json configs as bench workloads.  The default (and the only one the driver times) is the configuration the
# headline metric is quoted on; the others are for `python bench.py --workload ...` measurements recorded in profiles/.
WORKLOADS = {
    "spiral800": dict(H=800, W=800, level=7, code=32, kw=RENDER_KW, name="spiral_800x800_icosphere_V163842_F32_K8"),
    # config 2: "DTU scan63 full-res spiral" = 1600 x 1200 frames of the same scene
    "scan63_full": dict(H=1200, W=1600, level=7, code=32, kw=RENDER_KW, name="spiral_1600x1200_icosphere_V163842_F32_K8"),
    # config 3: "8-NN 256-d vertex codes", 800 x 800
    "codes256": dict(H=800, W=800, level=7, code=256, kw=RENDER_KW, name="spiral_800x800_icosphere_V163842_F256_K8"),
    # config 5: 2.6 M vertices, 256 samples per ray (image size from --image, default 4096 x 4096 split in bands)
    "big": dict(H=4096, W=4096, level=9, code=32,
                kw=dict(RENDER_KW, N_samples=128, N_importance=128, N_upsample_iters=4),
                name="spiral_4096x4096_icosphere_V2621442_F32_K8_256spp"),
}


def set_workload(name, image=0):
    global H, W, MESH_LEVEL, RENDER_KW, CODE_DIM, WORKLOAD_NAME, FLOP_GEO, FLOP_JVP, FLOP_COL
    w = WORKLOADS[name]
    H, W, MESH_LEVEL, RENDER_KW, CODE_DIM, WORKLOAD_NAME = w["H"], w["W"], w["level"], dict(w["kw"]), w["code"], w["name"]
    if image:
        H = W = int(image)
        WORKLOAD_NAME = WORKLOAD_NAME.replace("4096x4096", f"{H}x{W}").replace("800x800", f"{H}x{W}")
    kg, kc = 17 + 5 * CODE_DIM, 3 + 17 + 27 + 5 * CODE_DIM
    FLOP_GEO = 2 * (kg * 256 + 2 * 256 * 256 + 256)
    FLOP_JVP = 2 * (17 * 256 + 2 * 256 * 256 + 256)
    FLOP_COL = 2 * (kc * 256 + 3 * 256 * 256 + 3 * 256)


# algorithmic work per point (SURVEY.md section 8d; reference dims, no padding, each MAC counted once)
FLOP_GEO = 2 * (177 * 256 + 2 * 256 * 256 + 256)          # 353 280
FLOP_JVP = 2 * (17 * 256 + 2 * 256 * 256 + 256)           # 271 360 extra for the tangent rows
FLOP_COL = 2 * (207 * 256 + 3 * 256 * 256 + 3 * 256)      # 500 736
BYTES_KNN = 12 + 8 * 24                                   # 204 B per KNN query (xyz + 8 x (vertex + indicator))


def host_cores():
    """Physical cores of the host: MKL / OpenMP run the oracle fastest at one thread per physical core (measured on the
    GPU box: 210 rays/s at 64 threads, 39-50 rays/s at 128 hyper-threads)."""
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
        if n:
            return int(n)
    except Exception:
        pass
    return max(1, (os.cpu_count() or 2) // 2)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            d = json.load(open(path))
            return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d["bf16_tflops"]),
                    "bf16_tflops_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                    "source": "measured"}
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []
        self.thread = None
        self.first = 0

    def wait_ready(self, timeout: float = 3.0):
        """Block until nvidia-smi has delivered its first sample (its start-up is over) or `timeout` seconds passed."""
        t0 = time.perf_counter()
        while self.proc is not None and not self.lines and time.perf_counter() - t0 < timeout:
            time.sleep(0.02)

    def mark(self):
        """Start of the timed region: samples taken before (while nvidia-smi was starting up) are dropped."""
        self.first = len(self.lines)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=lambda: [self.lines.append(ln) for ln in self.proc.stdout], daemon=True)
        self.thread.start()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines[self.first:]:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def build_inputs(n_frames: int):
    cfg = synth.ModelConfig(geometry_dim=CODE_DIM, color_dim=CODE_DIM)
    mesh = synth.icosphere_mesh(MESH_LEVEL, seed=0)
    sd = synth.make_state_dict(mesh, cfg, seed=1)
    frames = [synth.frame_rays(H, W, view=v, n_views=90) for v in range(n_frames)]
    return cfg, mesh, sd, frames


def cpu_oracle_rate(cfg, mesh, sd, o, d, n_rays: int, repeats: int = 1):
    """rays/s of the oracle port (reference algorithm, torch CPU fp32, cKDTree exact KNN) on a strided ray sample."""
    torch.set_num_threads(host_cores())
    from oracle import render as orender
    from oracle.field import FieldOracle
    f = FieldOracle(mesh.vertices, sd, cfg)
    sel = torch.linspace(0, o.shape[0] - 1, n_rays).long()
    oo, dd = o[sel].contiguous(), d[sel].contiguous()
    orender.volume_render(oo[:64], dd[:64], f, rayschunk=4096, **RENDER_KW)  # builds the kd-tree, warms MKL
    best = None
    for _ in range(repeats):
        t = time.perf_counter()
        orender.volume_render(oo, dd, f, rayschunk=4096, **RENDER_KW)
        dt = time.perf_counter() - t
        best = dt if best is None else min(best, dt)
    return n_rays / best, best


def run_reference(args, rank, world):
    """`--impl reference`: the reference algorithm's own CPU path (oracle port; the reference is Python and cannot
    travel to the GPU box, see DESIGN.md), all host threads, bounded sample per step."""
    if rank != 0:
        return
    # all the host cores the box has (torchrun exports OMP_NUM_THREADS=1 to every rank: override it)
    torch.set_num_threads(host_cores())
    cfg, mesh, sd, frames = build_inputs(1)
    o, d = frames[0]
    n = args.ref_rays
    from oracle import render as orender
    from oracle.field import FieldOracle
    f = FieldOracle(mesh.vertices, sd, cfg)
    sel = torch.linspace(0, o.shape[0] - 1, n).long()
    oo, dd = o[sel].contiguous(), d[sel].contiguous()
    for _ in range(max(1, min(args.warmup, 1))):
        orender.volume_render(oo[:128], dd[:128], f, rayschunk=4096, **RENDER_KW)
    t = time.perf_counter()
    for _ in range(args.steps):
        orender.volume_render(oo, dd, f, rayschunk=4096, **RENDER_KW)
    dt = time.perf_counter() - t
    val = n * args.steps / dt
    cores = torch.get_num_threads()
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong" if (args.frames_per_step == 1 and world > 1) else "weak", "vs_baseline": None,
        "dtype": "fp32", "data": "synthetic", "config": workload_config(n),
        "cpu_baseline": {"value": val, "unit": "rays/s", "cores": cores, "kind": "port",
                         "sample": f"{n} rays strided over the 800x800 frame per step (oracle port of the reference "
                                   f"renderer, torch CPU fp32 + scipy cKDTree exact KNN, os.cpu_count()={os.cpu_count()})"},
        "e2e": {"value": val, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_config(rays_per_step):
    return {"workload": WORKLOAD_NAME, "image": [H, W], "rays_per_step": rays_per_step,
            "mesh_vertices": 10 * 4 ** MESH_LEVEL + 2, "vertex_code_dim": CODE_DIM, "knn_k": 8,
            "N_samples": RENDER_KW.get("N_samples", 64), "N_importance": RENDER_KW.get("N_importance", 64),
            "render": RENDER_KW,
            "l2": "inputs larger than L2: every step renders a different spiral view and streams ~12 GB of per-sample "
                  "scratch per frame (126 MB L2)"}


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(out, path):
    """Write the outputs of one step as ``path/<name>.npy`` (float32).  Above DUMP_BYTES in all, the same fixed, seeded
    sample of rays (ascending ray order) is taken from every array, so that two builds can be compared array for array."""
    os.makedirs(path, exist_ok=True)
    arrays = {k: v.detach().float().cpu() for k, v in out.items()}
    n = next(iter(arrays.values())).shape[0]
    per_ray = sum(v[0].numel() * 4 for v in arrays.values())
    keep = (DUMP_BYTES - 4096) // per_ray
    if keep < n:
        sel = torch.sort(torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep])[0]
        arrays = {k: v[sel] for k, v in arrays.items()}
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), v.numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--engine", default=DEFAULT_ENGINE, choices=["tcgen05", "fp32", "tcgen05_f16"],
                    help="MLP engine: tcgen05_f16 = fp16x3 operands (default), tcgen05 = 3xTF32, fp32 = CUDA cores")
    ap.add_argument("--workload", default="spiral800", choices=sorted(WORKLOADS) + ["train"],
                    help="spiral800 = the headline configuration (default, the one the driver times); scan63_full / "
                         "codes256 / big = BASELINE configs 2 / 3 / 5; train = config 4 (512 rays per GPU per step)")
    ap.add_argument("--image", type=int, default=0, help="override the (square) image size of the workload")
    ap.add_argument("--shard", default="auto", choices=["auto", "frame", "rays"],
                    help="multi-GPU partition of a step: whole frames per rank (when frames-per-step is a multiple of the "
                         "world size) or block-cyclic blocks of 128 rays of the pooled frames")
    ap.add_argument("--chunk", type=int, default=0, help="rays per kernel chunk (0 = library default)")
    ap.add_argument("--ref-rays", type=int, default=1024, help="rays per step of the CPU reference arm")
    ap.add_argument("--cpu-rays", type=int, default=1536, help="rays of the cpu_baseline sample (0 = skip)")
    ap.add_argument("--simulate-world", type=int, default=1,
                    help="(diagnostic, 1 GPU) render only rank 0's block-cyclic share of an N-way split and print the "
                         "per-rank time: predicts N-GPU throughput without N GPUs; not a bench value")
    ap.add_argument("--frames-per-step", type=int, default=0,
                    help="spiral frames rendered per step, their rays pooled and block-cyclic-sharded over the ranks "
                         "(default: one per GPU = fixed work per GPU, 'weak'; 1 = single-frame latency, 'strong')")
    ap.add_argument("--tune", action="store_true", help="(diagnostic) with --simulate-world 1: print per-class times only")
    ap.add_argument("--all-samples", action="store_true",
                    help="evaluate colour / nabla at every sample like the reference does, instead of only where the "
                         "visibility weight is non-zero (bit-identical outputs either way)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (rgb, depth_volume, mask_volume, "
                         "normals_volume) as DIR/<name>.npy, float32; a fixed sample of rays above 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.impl != "ours" or args.workload == "train" or args.simulate_world > 1 or args.tune):
        ap.error("--dump-outputs writes the outputs of the timed rendering steps: not with --impl reference, "
                 "--workload train, --simulate-world or --tune")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.workload == "train":
        import bench_train
        bench_train.main(args, rank, world, local_rank)
        return
    set_workload(args.workload, args.image)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist
    import neumesh_b200 as nb
    from neumesh_b200 import _lib, parallel
    from neumesh_b200.renderer import render_fused

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    sim = max(1, args.simulate_world)                # single-GPU what-if: render only rank 0's share of a `sim`-way split
    fps = 1 if (sim > 1 or args.tune) else (args.frames_per_step or world)
    scaling = "strong" if (fps == 1 and world > 1) else "weak"
    n_steps_in = max(1, min(args.warmup + args.steps, 90 // fps))      # distinct step inputs (90 spiral views)
    cfg, mesh, sd, views = build_inputs(n_steps_in * fps)
    frames = [(torch.cat([views[i * fps + j][0] for j in range(fps)]), torch.cat([views[i * fps + j][1] for j in range(fps)]))
              for i in range(n_steps_in)]
    del views
    model = nb.NeuMesh(nb.MeshGrid(mesh, dev), mlp_engine=args.engine, **cfg.model_kwargs())
    model.load_state_dict(sd)
    model = model.to(dev).eval()
    n_rays = H * W * fps                             # rays per step: `fps` consecutive spiral frames, pooled
    # partition of a step over the ranks: whole frames when there is at least one per rank (a rank's Morton-ordered
    # rays then belong to ONE camera pose - pooling blocks of eight different poses made the per-rank octree walks 30 %
    # slower at 8 GPUs in round 1), block-cyclic blocks of 128 rays otherwise (single-frame latency mode)
    by_frame = (args.shard == "frame" or (args.shard == "auto" and fps % world == 0 and fps >= world)) and sim == 1 \
        and world > 1 and fps % world == 0
    if by_frame:
        per = (fps // world) * H * W
        sl = torch.arange(rank * per, (rank + 1) * per)
        n_mine = per
    else:
        sl = parallel.shard_indices(n_rays, rank, world * sim)   # block-cyclic: every rank gets the same hit / miss mix
        n_mine = parallel.shard_count(n_rays, rank, world * sim)
    host = [(o[sl].contiguous().pin_memory(), d[sl].contiguous().pin_memory()) for o, d in frames]
    resident = [(o.to(dev), d.to(dev)) for o, d in host]
    chunk = args.chunk or None

    def step_resident(i, skip=None):
        o, d = resident[i % len(resident)]
        part = render_fused(o, d, model, chunk=chunk, skip_dead_samples=(not args.all_samples) if skip is None else skip,
                            **RENDER_KW)
        if sim > 1:
            return part
        if by_frame:
            return parallel.gather_image_contiguous(part, world)
        return parallel.gather_image(part, n_rays, rank, world)

    if sim > 1 or args.tune:
        assert world == 1, "--simulate-world is a single-GPU diagnostic"
        with torch.no_grad():
            for i in range(args.warmup):
                step_resident(i)
            torch.cuda.synchronize()
            _lib.profile_enable(True)
            _lib.profile_collect()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(args.steps):
                step_resident(args.warmup + i)
            e1.record()
            torch.cuda.synchronize()
            prof = _lib.profile_collect()
        ms = e0.elapsed_time(e1) / args.steps
        print(json.dumps({"diagnostic": "simulate_world", "world": sim, "rays_rank0": n_mine, "ms_per_step_rank0": ms,
                          "predicted_rays_per_s": n_rays / (ms * 1e-3),
                          "kernels_ms": {k: v["ms"] / args.steps for k, v in prof.items() if v["launches"]}}), flush=True)
        return

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        # the clock sampler (one long-running `nvidia-smi -lms`) starts BEFORE the warm-up: its start-up (NVML initialisation)
        # takes driver locks for a few hundred ms and must not fall into the timed region; only samples from the timed
        # region are reported
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
            sampler.wait_ready()
        for i in range(args.warmup):
            step_resident(i)
        barrier()

        # ---------------- timed region: inputs resident in HBM ----------------
        _lib.profile_enable(True)
        _lib.profile_collect()
        launches0 = _lib.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        sampler.mark()
        e0.record()
        for i in range(args.steps):
            out = step_resident(args.warmup + i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        clocks = sampler.stop() if rank == 0 else None
        launches = _lib.launch_count() - launches0
        prof = _lib.profile_collect()
        _lib.profile_enable(False)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms_total = float(ms.item())
        if args.dump_outputs and rank == 0:
            dump_outputs(out, args.dump_outputs)

        # ---------------- same frames with every sample evaluated (reference-style work), for transparency ----------------
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        step_resident(0, skip=False)
        barrier()
        g0.record()
        for i in range(args.steps):
            step_resident(args.warmup + i, skip=False)
        g1.record()
        barrier()
        ms3 = torch.tensor([g0.elapsed_time(g1)], device=dev)
        if world > 1:
            dist.all_reduce(ms3, op=dist.ReduceOp.MAX)
        ms_all = float(ms3.item())

        # ---------------- end to end through the public API with host buffers ----------------
        rgb_host = torch.empty(n_rays, 3).pin_memory()
        depth_host = torch.empty(n_rays).pin_memory()

        def step_e2e(i):
            o_h, d_h = host[i % len(host)]
            o = o_h.to(dev, non_blocking=True)
            d = d_h.to(dev, non_blocking=True)
            if world == 1 and not args.all_samples:
                rgb, depth, _ = nb.volume_render(o, d, model, detailed_output=False, **RENDER_KW)
            elif by_frame:
                part = render_fused(o, d, model, chunk=chunk, skip_dead_samples=not args.all_samples, **RENDER_KW)
                full = parallel.gather_image_contiguous(part, world)
                rgb, depth = full["rgb"], full["depth_volume"]
            else:
                full = parallel.render_sharded_local(o, d, model, n_rays, rank, world, chunk=chunk,
                                                     skip_dead_samples=not args.all_samples, **RENDER_KW)
                rgb, depth = full["rgb"], full["depth_volume"]
            if rank == 0:
                rgb_host.copy_(rgb, non_blocking=True)
                depth_host.copy_(depth, non_blocking=True)

        step_e2e(0)
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for i in range(args.steps):
            step_e2e(args.warmup + i)
        f1.record()
        barrier()
        ms2 = torch.tensor([f0.elapsed_time(f1)], device=dev)
        if world > 1:
            dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
        ms_e2e = float(ms2.item())

    if rank == 0:
        peaks = measured_peaks()
        value = n_rays * args.steps / (ms_total * 1e-3)
        e2e_val = n_rays * args.steps / (ms_e2e * 1e-3)
        # ---- per-kernel-class device time of THIS rank over the timed region ----
        kern = {}
        for k, v in prof.items():
            if v["launches"]:
                kern[k] = {"ms_per_step": v["ms"] / args.steps, "launches_per_step": v["launches"] / args.steps,
                           "points_per_step": v["points"] / args.steps}
        flops = {"geo": FLOP_GEO, "geo_jvp": FLOP_GEO + FLOP_JVP, "color": FLOP_COL}
        for k, fl in flops.items():
            if k in kern and kern[k]["ms_per_step"] > 0:
                kern[k]["tflops_algorithmic"] = kern[k]["points_per_step"] * fl / (kern[k]["ms_per_step"] * 1e-3) / 1e12
        for k in ("knn", "bound_scan", "knn_list"):
            if k in kern and kern[k]["ms_per_step"] > 0:
                kern[k]["gbs_algorithmic"] = kern[k]["points_per_step"] * BYTES_KNN / (kern[k]["ms_per_step"] * 1e-3) / 1e9
        mlp = [k for k in ("geo", "geo_jvp", "color") if k in kern]
        walk = [k for k in ("knn", "knn_list", "bound_scan") if k in kern]
        if mlp:   # the three instantiations of the ONE tcgen05 kernel template, taken together
            tot_ms = sum(kern[k]["ms_per_step"] for k in mlp)
            tot_fl = sum(kern[k]["points_per_step"] * flops[k] for k in mlp)
            kern["mlp_tc"] = {"ms_per_step": tot_ms, "launches_per_step": sum(kern[k]["launches_per_step"] for k in mlp),
                              "points_per_step": sum(kern[k]["points_per_step"] for k in mlp),
                              "tflops_algorithmic": tot_fl / (tot_ms * 1e-3) / 1e12}
            mlp = mlp + ["mlp_tc"]
        kname = {"geo": "mlp_tc_kernel<0> (geometry MLP)", "geo_jvp": "mlp_tc_kernel<1> (geometry MLP + tangent rows)",
                 "color": "mlp_tc_kernel<2> (colour MLP)", "mlp_tc": "mlp_tc_kernel<0|1|2> (tcgen05 field MLPs, all "
                 "instantiations)", "knn": "knn_rays_kernel (8-NN walk + mesh distance, ray-ordered)",
                 "knn_list": "knn_lists_kernel (8-NN walk + mesh distance, live samples)",
                 "bound_scan": "bound_dir_kernel<false|true> (bounded near/far: front-to-back + back-to-front scans)"}

        def tensor_roofline(k):
            peak = peaks["bf16_tflops_sustained"]
            ach = kern[k]["tflops_algorithmic"]
            split = ("every MAC is issued 3x as kind::f16 (fp16x3 split operands, fp32-accurate; needed for the 1e-4 / 1e-5 "
                     "parity bar), so the ceiling of this fraction is 1/3" if args.engine == "tcgen05_f16" else
                     "every MAC is issued 3x as kind::tf32 (3xTF32 split) and TF32 runs at half the bf16 rate, so the "
                     "ceiling of this fraction is 1/6")
            return {"bound": "tensor", "kernel": kname[k], "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                    "frac": ach / peak, "traffic": traffic_of(k),
                    "peak_source": f"{peaks['source']} dense bf16 cuBLAS, sustained",
                    "avg_launch_ms": kern[k]["ms_per_step"] / kern[k]["launches_per_step"],
                    "ms_per_step": kern[k]["ms_per_step"],
                    "note": "achieved = algorithmic fp32-equivalent FLOPs (each MAC once, reference dims) / device time "
                            "of the kernel class; " + split}

        def hbm_roofline(k):
            ach = kern[k]["gbs_algorithmic"]
            return {"bound": "hbm", "kernel": kname[k], "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": ach / peaks["hbm_gbs"], "traffic": traffic_of(k),
                    "peak_source": f"{peaks['source']} copy bandwidth",
                    "avg_launch_ms": kern[k]["ms_per_step"] / kern[k]["launches_per_step"],
                    "ms_per_step": kern[k]["ms_per_step"],
                    "note": "achieved = 204 algorithmic bytes per query (xyz + 8 x (vertex + indicator)) x queries / "
                            "device time.  The octree index (5.9 MB) is L2-resident and the walk is a divergent, "
                            "latency-bound pointer chase (ncu: DRAM < 1 %, SIMT efficiency 6-8 of 32 lanes, "
                            "long_scoreboard dominant): HBM bandwidth is the nominal roofline for a gather, not the "
                            "binding limit here"}

        traffic_tab = {}
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            try:
                traffic_tab = json.load(open(tpath))
            except Exception:
                traffic_tab = {}

        def traffic_of(k):
            """DRAM bytes per launch: ncu-measured bytes per processed point x points per launch of this run."""
            tab = traffic_tab.get("bytes_per_point", {})
            if k == "mlp_tc":
                parts = [kk for kk in ("geo", "geo_jvp", "color") if kk in kern and kk in tab]
                if not parts:
                    return None
                return sum(tab[kk] * kern[kk]["points_per_step"] for kk in parts) / kern[k]["launches_per_step"]
            if k == "walk":
                parts = [kk for kk in ("knn", "knn_list", "bound_scan") if kk in kern]
                vals = [traffic_of(kk) for kk in parts]
                if any(v is None for v in vals):
                    return None
                return sum(v * kern[kk]["launches_per_step"] for v, kk in zip(vals, parts)) / kern[k]["launches_per_step"]
            bpp = tab.get("knn" if k == "knn_list" else k)
            if bpp is None or k not in kern or not kern[k]["launches_per_step"]:
                return None
            return bpp * kern[k]["points_per_step"] / kern[k]["launches_per_step"]

        if walk:   # the three octree-walk kernels share knn_walk.cuh: one class, like the MLP instantiations
            tot_ms = sum(kern[k]["ms_per_step"] for k in walk)
            tot_pts = sum(kern[k]["points_per_step"] for k in walk)
            kern["walk"] = {"ms_per_step": tot_ms, "launches_per_step": sum(kern[k]["launches_per_step"] for k in walk),
                            "points_per_step": tot_pts, "gbs_algorithmic": tot_pts * BYTES_KNN / (tot_ms * 1e-3) / 1e9}
            kname["walk"] = "knn_rays_kernel + knn_lists_kernel + bound_dir_kernel (exact 8-NN octree walks, all)"
            walk = walk + ["walk"]
        roofline = None
        secondary = None
        allk = mlp + walk
        if allk:
            # the two kernel CLASSES of the frame: every tcgen05 MLP instantiation together, every octree walk together
            cls = [k for k in ("mlp_tc", "walk") if k in kern]
            cls.sort(key=lambda k: -kern[k]["ms_per_step"])
            mk = lambda k: tensor_roofline(k) if k in mlp else hbm_roofline(k)   # noqa: E731
            roofline = mk(cls[0])
            secondary = mk(cls[1]) if len(cls) > 1 else None
            roofline["by_class"] = {k: mk(k) for k in allk}
            for v in roofline["by_class"].values():
                v.pop("note", None)
            walk_issue = traffic_tab.get("walk_issue")
            if walk_issue and "walk" in kern:
                # honest second roofline of the latency / issue-bound walks: warp instructions per query from the ncu
                # capture of this very kernel x queries per second, against the SMs' issue rate at the sampled clock
                sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
                # queries that are really walked: the ray-ordered and the live-list kernels (the bound scan's nominal
                # 256 samples per ray are mostly decided by the certificate grid without a walk)
                qk = [k for k in ("knn", "knn_list") if k in kern]
                qps = sum(kern[k]["points_per_step"] for k in qk) / (sum(kern[k]["ms_per_step"] for k in qk) * 1e-3)
                peak = 148 * 4 * sm_mhz * 1e6
                tgt = roofline if cls[0] == "walk" else secondary
                tgt["issue_slots"] = {"warp_inst_per_query": walk_issue["warp_inst_per_query"],
                                      "active_lanes_per_inst": walk_issue["active_lanes_per_inst"],
                                      "achieved_warp_inst_per_s": qps * walk_issue["warp_inst_per_query"],
                                      "peak_warp_inst_per_s": peak,
                                      "frac": qps * walk_issue["warp_inst_per_query"] / peak,
                                      "kernels": "knn_rays_kernel + knn_lists_kernel",
                                      "note": "share of the SMs' warp-instruction issue slots the walks use (ncu "
                                              "issue-active 68-72 %); only ~10 of 32 lanes are active per issued "
                                              "instruction, so the USEFUL fraction is ~0.3 x this",
                                      "source": walk_issue.get("source", "profiles/")}
        cpu = None
        if world == 1 and args.cpu_rays > 0:
            rate, secs = cpu_oracle_rate(cfg, mesh, sd, frames[0][0], frames[0][1], args.cpu_rays)
            cpu = {"value": rate, "unit": "rays/s", "cores": torch.get_num_threads(), "kind": "port",
                   "sample": f"{args.cpu_rays} rays strided over frame 0 ({secs:.1f} s; oracle port of the reference "
                             f"renderer: torch CPU fp32 + scipy cKDTree exact KNN; os.cpu_count()={os.cpu_count()})"}
        bo = n_mine * 24
        bi = n_rays * 16
        line = {
            "metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None,
            "dtype": {"tcgen05": "fp32 (MLPs: 3xTF32 tcgen05, fp32 accumulate)",
                      "tcgen05_f16": "fp32 (MLPs: fp16x3 split operands on tcgen05 kind::f16, fp32 accumulate; sdf error "
                                     "vs float64 equal to plain fp32)"}.get(args.engine, "fp32"),
            "data": "synthetic", "config": {**workload_config(n_rays), "frames_per_step": fps,
                                            "parallelism": (f"whole-frame shard x{world} + all_gather" if by_frame else
                                                            f"block-cyclic ray-shard x{world} + all_gather"),
                                            "mlp_engine": args.engine,
                                            "skip_dead_samples": not args.all_samples},
            "e2e": {"value": e2e_val, "unit": "rays/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": bo, "d2h_bytes_per_step": bi,
                    "api": "neumesh_b200.volume_render on pinned host rays; rgb + depth read back to pinned host"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "roofline_secondary": secondary,
            "kernels": kern,
            "all_samples": {"value": n_rays * args.steps / (ms_all * 1e-3), "unit": "rays/s",
                            "ms_per_step": ms_all / args.steps,
                            "note": "same frames with colour / nabla evaluated at EVERY sample as the reference does "
                                    "(skip_dead_samples=False); outputs are bit-identical to the default path, which "
                                    "evaluates them only where the visibility weight is not exactly 0"},
            "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
