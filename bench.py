#!/usr/bin/env python
"""bench.py -- headline benchmark of the path-tracing hot path (BASELINE.json metric:
Msamples/s = path segments, i.e. trace_ray invocations, per second).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path
                                                             # (rpt-restated C++ oracle: the
                                                             # reference is Rust, no rustc here)

A "step" is one pass of Renderer::sample over one batch: the BASELINE configs[1] workload,
Cornell box 800x800, 512 spp per GPU, max_bounces 6.  At N GPUs the image gets 512*N spp and every
GPU renders 1/N of the 16x8 pixel tiles (per-GPU work fixed => weak scaling) into a compact
tile-major buffer; ONE all-gather of those shards (NCCL) and a fixed permutation assemble the float3
image on every rank.  Prints ONE JSON line on rank 0.

Besides the headline (`value`, `e2e`, `roofline`, `cpu_baseline`) the line carries `secondary`: the two BASELINE
configs quoted on 8 GPUs -- dragon (1920x1080, 1024 spp, max_bounces 2) and glass (1920x1080, 4096 spp,
max_bounces 12) -- rendered ONCE each at their full size with the pixel tiles split over the N ranks (fixed total
work => strong scaling), device-timed, with the HBM roofline of the BVH traffic on the dragon.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import socket
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "Msamples/s (path segments = trace_ray invocations per second)"
UNIT = "Msamples/s"
CPU_SPP_PER_STEP = 16  # samples per pixel of one CPU-arm step (full resolution, full max_bounces)
KEYS = ["segments", "rays", "node_visits", "tri_tests", "mesh_hits", "env_lookups", "object_tests", "bvh_node_visits", "bvh_tri_tests"]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="cornell",
                    choices=["sphere", "cornell", "teapot", "dragon", "glass",
                             "fractal_spheres", "fractal_teapots", "monomial_glass", "dragon_knot"],  # the last four: exploration only
                    help="default = the BASELINE configs[1] workload; anything else is for exploration / profiling")
    ap.add_argument("--spp", type=int, default=0, help="override samples per pixel per GPU (exploration only)")
    ap.add_argument("--engine", default="auto", choices=["auto", "megakernel", "wavefront"], help="rptb_engine (exploration only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the dragon / glass strong-scaling block")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the image the last one assembled to DIR/image.npy "
                         "(float32, height x width x 3), to compare two builds on the same inputs")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes what the native arm computed; the reference arm has no such output")
    return args


def workload(name: str, spp_override: int = 0):
    from rpt_b200 import scenes

    cfg = (scenes.CONFIGS[name] if name in scenes.CONFIGS else scenes.EXTRA_CONFIGS[name])()
    if spp_override:
        cfg.spp = spp_override
    return cfg


def config_dict(cfg, world: int):
    """The same dictionary in both arms (the CPU arm renders a bounded sample of exactly this workload)."""
    return {
        "workload": "%s %dx%d, %d spp per GPU (%d total), max_bounces %d; %s" % (
            cfg.name, cfg.width, cfg.height, cfg.spp, cfg.spp * world, cfg.max_bounces, cfg.note),
        "scene": cfg.name,
        "width": cfg.width,
        "height": cfg.height,
        "spp_per_gpu": cfg.spp,
        "spp_total": cfg.spp * world,
        "max_bounces": cfg.max_bounces,
        "parallelism": "pixel tiles 16x8 round-robin over %d GPU(s); one all-gather of the ranks' own tiles (1/N of the float3 image each)" % world,
        "rng": "Philox4x32-10 keyed (seed=1, pixel, sample)",
        "cache": "L2 flushed between timed steps (256 MiB memset); the Cornell scene itself is 4 KiB and cache-resident by nature",
    }


# ------------------------------------------------------------------ clocks ------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, ngpus: int):
        self.ngpus = ngpus
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                idx = int(f[0])
                if idx >= self.ngpus:
                    continue
                sm.append(float(f[1]))
                smax.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(smax), "power_w_max": max(power), "samples": len(sm),
                "reasons": sorted(reasons)}


# ------------------------------------------------------------------ roofline ----------
def algorithmic_bytes(stats: dict, pixels: int) -> float:
    """SURVEY 8(d) per-unit figures with this repo's device layout (DESIGN.md section 5):
    64 B object record per Shape::intersect dispatch; the structure that was traversed -- 64 B per BVH node fetched
    (both child boxes) and 48 + 4 B per triangle tested in a BVH leaf, or 8 B per kd node and 4 + 48 B per triangle
    test on a kd-tree scene; 36 B vertex normals per mesh hit; 32 B material per segment; 64 B (4 texels x 16 B)
    per HDRI lookup; 12 B per pixel written."""
    return (64.0 * stats["object_tests"] + 8.0 * stats["node_visits"] + 52.0 * stats["tri_tests"]
            + 64.0 * stats.get("bvh_node_visits", 0) + 52.0 * stats.get("bvh_tri_tests", 0)
            + 36.0 * stats["mesh_hits"] + 32.0 * stats["segments"] + 64.0 * stats["env_lookups"] + 12.0 * pixels)


BYTES_MODEL = ("64*object_tests + 64*bvh_node_visits + 52*bvh_tri_tests + 8*node_visits + 52*tri_tests + 36*mesh_hits + "
               "32*segments + 64*env_lookups + 12*pixels (counters of the structure that rendered the step: collect_stats = 1)")


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            d = json.load(open(path))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)", float(d.get("sm_max_mhz", 1965.0))
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)", 1965.0


def ncu_record(workload_name: str):
    """Per-launch figures of the dominant kernel from the committed `ncu --set full` capture of this round
    (profiles/ncu_kernels.json, written by tools/ncu_kernels_json.py): dram bytes, warp and thread instructions and
    the segments the captured launch traced -- the per-segment ratios are properties of the kernel."""
    try:
        rec = json.load(open(os.path.join(ROOT, "profiles", "ncu_kernels.json"))).get(workload_name)
        return rec if isinstance(rec, dict) else None
    except Exception:
        return None


# ------------------------------------------------------------------ CPU arm -----------
def host_cores():
    """Threads this process may really use: the scheduler affinity, capped by the cgroup CPU quota (a GPU box
    reports 128 CPUs and grants 16 of them)."""
    try:
        aff = len(os.sched_getaffinity(0))
    except AttributeError:
        aff = os.cpu_count() or 1
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        pass
    used = aff if quota is None else max(1, min(aff, int(quota + 0.5)))
    return used, aff, quota


def cpu_arm(cfg, steps: int, warmup: int, budget_s: float = None):
    """The CPU restatement of the same workload on all usable host threads: every step renders CPU_SPP_PER_STEP
    samples per pixel of the full-resolution image (the rate does not depend on spp).  With `budget_s`, stops early
    once that much time has been spent (cpu_baseline leg of the native arm)."""
    from oracle import oracle_py as orc
    from rpt_b200 import api

    flat = api.FlatScene(cfg.scene)
    osc = orc.OracleScene(flat)
    r = api.Renderer(cfg.scene, cfg.camera).width(cfg.width).height(cfg.height).max_bounces(cfg.max_bounces).seed(1)
    cores, aff, quota = host_cores()
    first = 0
    for _ in range(warmup):
        osc.render(cfg.camera, r.params(1, first), nthreads=cores)
        first += 1
    segs, t, done = 0, 0.0, 0
    for _ in range(steps):
        t0 = time.perf_counter()
        _, st = osc.render(cfg.camera, r.params(CPU_SPP_PER_STEP, first), nthreads=cores)
        t += time.perf_counter() - t0
        first += CPU_SPP_PER_STEP
        segs += st["segments"]
        done += 1
        if budget_s is not None and t >= budget_s:
            break
    value = segs / t / 1e6
    sample = ("%s %dx%d, max_bounces %d: %d step(s) of %d spp (of %d) at full resolution = %d segments in %.2f s; "
              "rpt-restated C++ f64 oracle, OpenMP over rows on %d threads (affinity %d, cgroup quota %s); rpt itself is Rust and "
              "cannot be built here" % (cfg.name, cfg.width, cfg.height, cfg.max_bounces, done, CPU_SPP_PER_STEP, cfg.spp, segs, t,
                                        cores, aff, "none" if quota is None else "%.1f" % quota))
    return {"value": value, "unit": UNIT, "cores": cores, "cores_affinity": aff, "cgroup_cpu_quota": quota, "kind": "port",
            "sample": sample, "steps": done, "seconds": t}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cfg = workload(args.workload, args.spp)
    res = cpu_arm(cfg, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * res["seconds"] / max(res["steps"], 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(cfg, args.gpus),
        "note": "CPU path (n_gpus is echoed, no GPU is used); each step is a bounded sample of the workload, see cpu_baseline.sample",
        "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "cores_affinity", "cgroup_cpu_quota", "kind", "sample")},
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


# ------------------------------------------------------------------ GPU arm -----------
def free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def run_native(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    import numpy as np
    import torch
    import torch.distributed as dist

    from rpt_b200 import _capi as capi
    from rpt_b200 import api
    from rpt_b200 import distributed as D

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if capi.lib().rptb_device_count() <= 0:
        raise SystemExit("bench.py: no CUDA device and rpt_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    cpu_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        # a barrier the waiting ranks sit in on the CPU: while rank 0 drives all N GPUs through ONE rptb_render_samples
        # call (e2e leg), an NCCL barrier kernel spinning on the other ranks' GPUs would time-slice against its kernels
        cpu_group = dist.new_group(backend="gloo")
    engine = {"auto": capi.ENGINE_AUTO, "megakernel": capi.ENGINE_MEGAKERNEL, "wavefront": capi.ENGINE_WAVEFRONT}[args.engine]
    stream = torch.cuda.Stream(dev)
    raw = stream.cuda_stream
    K, W = args.steps, args.warmup
    peak, peak_src, sm_max_mhz = measured_peaks()

    def barrier():
        if world > 1:
            dist.barrier()

    def cpu_barrier():
        if world > 1:
            dist.barrier(group=cpu_group)

    def allsum(vals, dtype=torch.int64):
        t = torch.tensor(vals, dtype=dtype, device=dev)
        if world > 1:
            dist.all_reduce(t)
        return t.tolist()

    def allmax(vals):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()

    class Job:
        """One workload on this rank: renderer, compact shard buffer, gather permutation."""

        def __init__(self, cfg, spp_total):
            self.cfg, self.spp_total = cfg, spp_total
            self.r = api.Renderer(cfg.scene, cfg.camera).width(cfg.width).height(cfg.height).max_bounces(cfg.max_bounces) \
                .seed(1).device(local).engine(engine)
            self.npix = cfg.width * cfg.height
            self.shard = torch.zeros(D.shard_tiles(cfg.width, cfg.height, 0, world) * 384, dtype=torch.float32, device=dev)
            self.perm = torch.from_numpy(D.gather_permutation(cfg.width, cfg.height, world)).to(dev)
            self.image = None

        def render(self, stats=None, collect_stats=0, spp=None):
            D.render_shard_device(self.r, spp or self.spp_total, self.shard, rank, world, 0, raw, stats=stats,
                                  collect_stats=collect_stats, compact=True)

        def assemble(self):
            self.image = D.gather_tiles(lambda rk, wd: self.shard, self.cfg.width, self.cfg.height, self.perm)

        def counters(self, spp=None):
            st = capi.Stats()
            self.render(st, 1, spp)
            mine = st.as_dict()
            tot = dict(zip(KEYS, [int(v) for v in allsum([mine[k] for k in KEYS])]))
            return tot, int(st.launches), int(st.engine)

        def close(self):
            self.r.close()

    with torch.cuda.stream(stream):
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        cfg = workload(args.workload, args.spp)
        job = Job(cfg, cfg.spp * world)
        flat = api.FlatScene(cfg.scene)
        npix = job.npix

        # un-timed statistics pass: exact segment count of one step + the traversal counters of what renders it
        total, launches_per_step, engine_used = job.counters()
        launches_per_step += (1 if world > 1 else 0) + 1  # + NCCL all-gather kernel, + torch's index_select (the permutation)

        def step(ev_mid=None):
            job.render()
            if ev_mid is not None:
                ev_mid.record()
            job.assemble()

        for _ in range(W):
            step()
        stream.synchronize()
        barrier()
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(K)]
        sampler = ClockSampler(world) if rank == 0 else None
        if sampler:
            sampler.start()
        t_wall = time.perf_counter()
        for i in range(K):
            flush.zero_()  # evict L2 between timed steps (outside the event pair)
            ev[i][0].record()
            step(ev[i][1])
            ev[i][2].record()
        stream.synchronize()
        barrier()
        t_wall = time.perf_counter() - t_wall
        clocks = sampler.stop() if sampler else None
        # per step: the slowest rank's kernel, the slowest rank's whole step (a rank's step includes waiting in the
        # collective for the slowest kernel), and the fastest rank's kernel (spread = content imbalance between shards)
        kern = [e[0].elapsed_time(e[1]) for e in ev]
        stepms = [e[0].elapsed_time(e[2]) for e in ev]
        kern_max = allmax(kern)
        step_max = allmax(stepms)
        kern_min = [-v for v in allmax([-v for v in kern])]
        step_ms = sum(step_max)
        kern_ms = sum(kern_max)
        image_mean = float(job.image.mean().item())
        if args.dump_outputs and rank == 0:  # every rank holds the whole image after the all-gather
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "image.npy"),
                    job.image.view(cfg.height, cfg.width, 3).cpu().numpy())

        # ---- e2e: the public call with HOST buffers, copies inside the timed region -----
        e2e = None
        if not args.no_e2e:
            host64 = np.empty((npix, 3), np.float64)
            cam = cfg.camera.to_c()
            devices = list(range(world))

            def e2e_step():
                # H2D: the flattened scene (host arrays -> HBM of every GPU); one call renders on all of them and leaves
                # the image in the caller's double buffer (D2H inside)
                ds = api.DeviceScene(flat, devices if world > 1 else local)
                try:
                    p = job.r.params(job.spp_total, 0, 0, 1)
                    capi.check(capi.lib().rptb_render_samples(ds.handle, C.byref(cam), C.byref(p),
                                                              host64.ctypes.data_as(capi.c_double_p), None), "rptb_render_samples")
                finally:
                    ds.close()

            stream.synchronize()
            barrier()
            torch.cuda.synchronize()
            cpu_barrier()
            e2e_s = 0.0
            if rank == 0:  # the fan-out over the N GPUs lives inside rptb_render_samples: one caller, the other ranks wait (on the CPU)
                e2e_step()  # warm-up
                t0 = time.perf_counter()
                for _ in range(K):
                    e2e_step()
                e2e_s = time.perf_counter() - t0
            cpu_barrier()
            if rank == 0:
                e2e = {
                    "value": total["segments"] * K / e2e_s / 1e6, "unit": UNIT,
                    "h2d_bytes_per_step": int(flat.host_bytes() + C.sizeof(capi.Camera) + C.sizeof(capi.RenderParams)) * world,
                    "d2h_bytes_per_step": int(npix * 3 * 4),
                    "ms_per_step": 1e3 * e2e_s / K,
                    "call": ("rptb_scene_create + rptb_render_samples(host double* out) + rptb_scene_destroy per step" if world == 1 else
                             "rptb_scene_create_multi(%d GPUs) + ONE rptb_render_samples(host double* out) + rptb_scene_destroy per step, "
                             "called by rank 0 (one host thread per GPU inside the library; the other ranks idle)" % world),
                    "timer": "host perf_counter around the K calls (each call returns with the image in host memory)",
                    "h2d_source": "pageable host arrays (cudaMemcpy inside rptb_scene_create*)",
                    "image_mean": float(host64.mean()),
                }

        # ---- secondary: BASELINE's 8-GPU configs at their own size, strong scaling ------------------------------
        secondary = None
        if args.workload == "cornell" and not args.no_secondary and not args.spp:
            secondary = {}
            for name in ("dragon", "glass"):
                scfg = workload(name)
                sj = Job(scfg, scfg.spp)  # the image gets scfg.spp samples however many ranks share it
                probe_spp = max(1, scfg.spp // 64)
                ctr, _, _ = sj.counters(probe_spp)   # counters per segment at reduced spp (they scale with the sample count)
                sj.render(spp=probe_spp)             # warm-up of the plain kernel
                sj.assemble()
                # ... and one un-timed render at the full size: the first full-size launch of a process is slower than the
                # ones after it (measured, tools/gpu_fullspp_repeat.py, two processes alike: dragon 1 688 / 1 709 then 1 821 /
                # 1 851, glass 20 787 / 20 562 then 21 233 / 21 209 Msamples/s; it is also the first launch that needs the
                # full set of chunk sums in scratch)
                sj.render()
                sj.assemble()
                stream.synchronize()
                barrier()
                e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                flush.zero_()
                st = capi.Stats()
                ssampler = ClockSampler(world) if rank == 0 else None
                if ssampler:
                    ssampler.start()
                e0.record()
                sj.render(st)  # collect_stats = 0: segments / rays only; the call returns when the kernel has finished
                e1.record()
                sj.assemble()
                e2.record()
                stream.synchronize()
                sclocks = ssampler.stop() if ssampler else None
                barrier()
                segs, rays = allsum([int(st.segments), int(st.rays)])
                t_step, t_kern = allmax([e0.elapsed_time(e2), e0.elapsed_time(e1)])
                scale = segs / max(ctr["segments"], 1)
                bytes_all = algorithmic_bytes({k: v * scale for k, v in ctr.items()}, sj.npix)
                ach = bytes_all / world / (t_kern / 1e3) / 1e9
                secondary[scfg.name] = {
                    "config": "%s %dx%d, %d spp total, max_bounces %d; %s" % (scfg.name, scfg.width, scfg.height, scfg.spp, scfg.max_bounces, scfg.note),
                    "scaling": "strong", "steps": 1, "warmup": "one %d-spp render + one full-size render" % probe_spp,
                    "value": segs / (t_step / 1e3) / 1e6, "unit": UNIT,
                    "ms_per_step": t_step, "kernel_ms_max_rank": t_kern, "segments": segs, "rays": rays,
                    "image_mean": float(sj.image.mean().item()), "device_scene_bytes": sj.r.device_scene().device_bytes(),
                    "clocks": sclocks,
                    "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                                 "algorithmic_bytes_per_launch": bytes_all / world, "bytes_model": BYTES_MODEL,
                                 "per_ray": {"bvh_nodes": ctr["bvh_node_visits"] / max(ctr["rays"], 1), "bvh_tris": ctr["bvh_tri_tests"] / max(ctr["rays"], 1),
                                             "objects": ctr["object_tests"] / max(ctr["rays"], 1)},
                                 "traffic": (lambda rec: None if not rec else rec["dram_bytes"] * segs / world / max(rec["segments"], 1))(ncu_record(scfg.name)),
                                 "note": "counters from a %d-spp pass of the counting variant of the same kernel, scaled by segments" % probe_spp},
                }
                sj.close()

    if rank == 0:
        value = total["segments"] * K / (step_ms / 1e3) / 1e6
        bytes_all = algorithmic_bytes(total, npix)  # summed over ranks (each writes its own pixels)
        kern_s = kern_ms / 1e3 / K
        achieved_hbm = bytes_all / world / kern_s / 1e9  # per GPU
        rec = ncu_record(cfg.name)
        sm_mhz = (clocks or {}).get("sm_mhz") or sm_max_mhz
        segs_per_gpu = total["segments"] / world
        hbm_view = {"achieved_algorithmic_gbs": achieved_hbm, "peak": peak, "unit": "GB/s", "frac_algorithmic": achieved_hbm / peak,
                    "peak_source": peak_src, "algorithmic_bytes_per_launch": bytes_all / world, "bytes_model": BYTES_MODEL,
                    "counters_per_step": total}
        if rec:
            traffic = rec["dram_bytes"] * segs_per_gpu / max(rec["segments"], 1)
            hbm_view["dram_frac"] = traffic / kern_s / 1e9 / peak
        else:
            traffic = None
        cache_resident = flat.host_bytes() < (32 << 20)
        if cache_resident and rec:
            # a scene that lives in L1/L2 is bound by instruction issue, not by HBM: thread-instructions per second against
            # 148 SMs x 128 FP32 lanes x the SM clock sampled during the run (the per-segment instruction count is the
            # kernel's, from this round's ncu capture)
            tinst = rec["thread_inst"] * segs_per_gpu / max(rec["segments"], 1)
            ach = tinst / kern_s / 1e9
            pk = 148 * 128 * sm_mhz * 1e6 / 1e9
            roofline = {"bound": "issue", "achieved": ach, "peak": pk, "unit": "Gthread-inst/s", "frac": ach / pk, "traffic": traffic,
                        "peak_source": "148 SMs x 128 lanes x %.0f MHz (median SM clock during the timed region)" % sm_mhz,
                        "thread_inst_per_segment": rec["thread_inst"] / max(rec["segments"], 1),
                        "lanes_per_warp_inst": rec["thread_inst"] / max(rec["inst"], 1),
                        "note": "the whole scene is cache resident (%d B): the HBM view below counts bytes L1/L2 serve" % flat.host_bytes(),
                        "hbm": hbm_view}
        else:
            roofline = {"bound": "hbm", "achieved": achieved_hbm, "peak": peak, "unit": "GB/s", "frac": achieved_hbm / peak, "traffic": traffic,
                        "peak_source": peak_src, "algorithmic_bytes_per_launch": bytes_all / world, "bytes_model": BYTES_MODEL,
                        "counters_per_step": total}
        roofline["kernel"] = ("rptb::render_kernel<float,16,false,FEAT> (megakernel: one launch per step, + chunk resolve)" if engine_used != 2 else
                              "rptb::wf_trace_kernel (+ wf_shade_kernel; wavefront engine: the duration is the whole step's kernels)")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": step_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": config_dict(cfg, world),
            "segments_per_step": total["segments"], "rays_per_step": total["rays"],
            "kernel_ms_per_step": kern_ms / K, "wall_s_timed_region": t_wall, "image_mean": image_mean,
            "step_breakdown_ms": {
                "kernel_slowest_rank": kern_ms / K, "kernel_fastest_rank": sum(kern_min) / K,
                "collective_and_assembly": (step_ms - kern_ms) / K,
                "note": "per step: max over ranks of the render kernel, its spread across ranks (shard content), and what the "
                        "all-gather + permutation add on top of the slowest kernel",
            },
            "clocks": clocks,
            "e2e": e2e,
            "gpu_launches": launches_per_step * K,
            "roofline": roofline,
        }
        if secondary:
            line["secondary"] = secondary
        if world == 1 and not args.no_cpu_baseline:
            res = cpu_arm(cfg, 8, 1, budget_s=12.0)
            line["cpu_baseline"] = {k: res[k] for k in ("value", "unit", "cores", "cores_affinity", "cgroup_cpu_quota", "kind", "sample")}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    job.close()
    return 0


def main():
    args = parse_args()
    # Exactly ONE line may reach stdout.  Libraries write there too (NCCL prints its version banner
    # to stdout when NCCL_DEBUG is set), so fd 1 is pointed at stderr for the whole run and the JSON
    # line goes to the saved descriptor.
    if args.impl == "native" and args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # convenience: re-launch under torchrun exactly like the driver does
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(free_port()), os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args)
    return run_native(args)


_REAL_STDOUT = None


def emit(line: dict) -> None:
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


if __name__ == "__main__":
    sys.exit(main())
