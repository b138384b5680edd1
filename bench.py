#!/usr/bin/env python
"""bench.py -- Msamples/s (paths x bounces) of the guided path tracer, one JSON line.

A "step" is one complete guided render (all training iterations + the final iteration, tree maintenance
included) of the workload through the C ABI of libppg_b200.so.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--scene cbox|kitchen|spaceship|torus]     our arm (one rank per GPU under torchrun for N > 1)
  python bench.py --impl reference ...                                                            the reference's CPU algorithm on the host cores

Default workload (BASELINE.json configs[1]): CBOX 1024x1024, default Mueller'17 parameters (sppPerPass 4, maxDepth 10,
rrDepth 10, strictNormals, nearest/nearest filters, sampleCombination automatic, sTreeThreshold 12000).  The reference quotes
it on a 60 s budget; Msamples/s is a rate, so a step uses an equal-spp budget instead (budgetType=spp, 252 spp = 63 passes =
iterations of 1,2,4,8,16,32 passes) so that a step takes a fraction of a second and the equal-spp image comparison of the
metric's second half (relMSE against a converged image, GPU vs the reference algorithm) is meaningful.  --budget-seconds runs
the literal time-budget configuration.  The other named scenes of BASELINE.json run with their XML settings at the BASELINE
resolutions: --scene kitchen (config 3, 1280x720), spaceship (config 4, 1920x1080), torus (config 5 stand-in, 1024x1024).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "practical-path-guiding_b200"))

import numpy as np  # noqa: E402

SCENES = {
    # name: (fixture or builtin, width, height, default spp budget of one step, description)
    "cbox": ("cbox", 1024, 1024, 252, "CBOX 1024x1024, default Mueller'17 params (sppPerPass=4, maxDepth=10, rrDepth=10, nearest/nearest, automatic, sTreeThreshold=12000)"),
    "kitchen": ("kitchen-improved", 1280, 720, 127, "KITCHEN 1280x720 with improvements (inversevar / stochastic / box / kl, sTreeThreshold=4000, sppPerPass=1), 1 414 391 triangles, 13 bitmap textures, sunsky"),
    "spaceship": ("spaceship-improved", 1920, 1080, 127, "SPACESHIP 1920x1080 with improvements (inversevar / stochastic / box / kl, sTreeThreshold=4000, sppPerPass=1), 457 560 triangles"),
    "torus": ("builtin:torus", 1024, 1024, 127, "TORUS stand-in 1024x1024 (glass cube around a diffuse torus: SDS caustics; the reference's asset is not bundled), sTreeThreshold=4000, sppPerPass=1"),
}


def load_scene(name, w=None, h=None):
    from ppg_b200.scene import SceneDesc
    fixture, W, H, _, _ = SCENES[name]
    w, h = w or W, h or H
    if fixture == "builtin:torus":
        from ppg_b200.builtin_scenes import torus_scene
        sc = torus_scene(w)
        return sc.with_film(w, h)
    return SceneDesc.load(os.path.join(ROOT, "scenes", fixture + ".npz")).with_film(w, h)


def host_cores():
    """Cores this process may actually use: the affinity mask, capped by a cgroup CPU quota (os.cpu_count() reports the machine)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for p in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(p).read().split()
            if p.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]))))
            else:
                q = int(txt[0]); per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, n)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json, torch copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def relmse(img, ref):
    """SURVEY 8d: mean over pixels of (img - ref)^2 / (ref^2 + 1e-3)."""
    img = np.asarray(img, np.float64); ref = np.asarray(ref, np.float64)
    return float(np.mean((img - ref) ** 2 / (ref ** 2 + 1e-3)))


def converged_reference(scene, w, h):
    """Converged image of the workload (tools/make_reference.py: the product at 32768 spp, float16), or None."""
    p = os.path.join(ROOT, "scenes", "ref", f"{scene}_{w}x{h}_ref.npy")
    return np.load(p).astype(np.float32) if os.path.exists(p) else None


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed regions (B200_PROFILING.md's clocks line). NVML is polled from a thread
    every 10 ms (nvidia-smi -lms needs >100 ms to start, longer than an 8-GPU timed region); nvidia-smi is the fallback."""

    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, index=0, uuid=None):
        self.index = index; self.uuid = uuid; self.rows = []; self.active = False; self.stopflag = False; self.thread = None; self.kind = None
        self.max_mhz = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if self.uuid:
                try:
                    h = pynvml.nvmlDeviceGetHandleByUUID(self.uuid if self.uuid.startswith("GPU-") else "GPU-" + self.uuid)
                except Exception:
                    h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))

            def poll():
                while not self.stopflag:
                    if self.active:
                        try:
                            self.rows.append((float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)), int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))))
                        except Exception:
                            pass
                    time.sleep(0.01)
            self.kind = "nvml"
            self.thread = threading.Thread(target=poll, daemon=True); self.thread.start()
            return
        except Exception:
            pass
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)

            def read():
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                for line in self.proc.stdout:
                    f = [x.strip() for x in line.split(",")]
                    if len(f) < 6 or not self.active:
                        continue
                    try:
                        mask = sum(self.REASONS[n] for n, v in zip(names, f[2:6]) if v.lower().startswith("active"))
                        self.rows.append((float(f[0]), mask)); self.max_mhz = float(f[1])
                    except ValueError:
                        pass
            self.kind = "nvidia-smi"
            self.thread = threading.Thread(target=read, daemon=True); self.thread.start()
            time.sleep(0.5)
        except Exception:
            self.kind = None

    def region(self, on):
        self.active = bool(on)

    def stop(self):
        self.stopflag = True; self.active = False
        if self.kind == "nvidia-smi":
            self.proc.terminate()
        if self.kind is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml and nvidia-smi unavailable"], "samples": 0}
        sm = [r[0] for r in self.rows]
        reasons = sorted(n for n, bit in self.REASONS.items() if any(r[1] & bit for r in self.rows))
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(sm), "source": self.kind}


def scene_props(args, sc, budget=None):
    props = dict(sc.integrator)
    if args.budget_seconds:
        props.update(budgetType="seconds", budget=str(args.budget_seconds))
    else:
        props.update(budgetType="spp", budget=str(budget if budget is not None else args.budget))
    return props


def workload_config(args, bounded=None):
    desc = SCENES[args.scene][4]
    c = {"workload": f"{desc}, " + (f"budgetType=seconds budget={args.budget_seconds}" if args.budget_seconds else
                                    f"budgetType=spp budget={args.budget}" + (" (equal-spp stand-in for the 60 s budget of BASELINE config 2)" if args.scene == "cbox" else "")),
         "scene": f"scenes/{SCENES[args.scene][0]}.npz" if not SCENES[args.scene][0].startswith("builtin") else "ppg_b200.builtin_scenes.torus_scene",
         "width": args.width, "height": args.height,
         "sharding": f"32x32 image blocks dealt round-robin in a scattered order over {args.gpus} rank(s); one NCCL allreduce of the D-tree sums per training iteration, enqueued on the render stream by the library",
         "l2": "inputs larger than L2: path state + vertex records of one pass-batch are ~1 GB, every kernel streams them once"}
    if bounded:
        c["bounded_sample"] = bounded
    return c


# ------------------------------------------------------------------------------------------- CPU arm

def cpu_run(args, w, h, budget, nthreads):
    """Times the CPU oracle (the reference algorithm: restated tracer; SD-tree compiled verbatim from the reference when
    oracle/_ref/libppg_oracle_ref.so travelled) on the host cores this process owns."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    kind = "ref" if O.have_ref() else "port"
    sc = load_scene(args.scene, w, h)
    props = dict(sc.integrator, budgetType="spp", budget=str(budget))
    o = O.Oracle(O.params_from_xml(props), sc, nthreads=nthreads, kind=kind)
    t = time.perf_counter()
    img, st = o.render()
    dt = time.perf_counter() - t
    o.close()
    return {"seconds": dt, "vertices": st["total_vertices"], "paths": st["total_paths"], "msamples": st["total_vertices"] / dt / 1e6,
            "kind": kind, "image": img, "stats": st, "w": w, "h": h, "budget": budget}


def cpu_sample_size(args):
    """The CPU arm runs the SAME configuration for CBOX (one step of 1024^2 / 252 spp is ~1.1 G vertices: 20 - 110 s on 128 - 8 cores).  The
    heavier scenes run a bounded sample (quarter resolution, fewer spp) of the same workload; said so in the line."""
    if args.scene == "cbox" and not args.cpu_bounded:
        return args.width, args.height, args.budget, True
    if args.scene == "cbox":
        return 512, 512, 60, False
    return max(64, args.width // 4), max(64, args.height // 4), min(args.budget, 63), False


def cpu_line_fields(r, cores, same):
    kind = "reference" if r["kind"] == "ref" else "port"
    sample = (f"{r['w']}x{r['h']}, budget {r['budget']} spp: {r['paths']} paths / {r['vertices']} vertices in {r['seconds']:.1f} s on {cores} threads "
              f"(CPU tracer restated from guided_path.cpp; SD-tree {'compiled verbatim from the reference' if kind == 'reference' else 'restated'}; OpenMP over 32x32 blocks); "
              + ("same configuration as the GPU arm" if same else "bounded sample of the GPU arm's workload"))
    return {"value": r["msamples"], "unit": "Msamples/s", "cores": cores, "kind": kind, "sample": sample, "same_config": bool(same)}


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cores()
    w, h, budget, same = cpu_sample_size(args)
    # one repetition of the full configuration takes 20 s (128 cores) to 2 min (8 cores): the step count is bounded by a time budget
    vals = []; t0 = time.perf_counter()
    for i in range(args.warmup + args.steps):
        if vals and time.perf_counter() - t0 > args.cpu_seconds:
            break
        r = cpu_run(args, w, h, budget, cores)
        if same or i >= args.warmup or args.warmup + args.steps == 1:
            vals.append(r)           # (a full-size repetition is never thrown away as warm-up: the first one already runs minutes of steady state)
    v = float(np.mean([r["msamples"] for r in vals]))
    ms = float(np.mean([r["seconds"] for r in vals]) * 1e3)
    cb = cpu_line_fields(vals[-1], cores, same)
    cb["value"] = v
    line = {
        "impl": "reference", "metric": "Msamples/sec (paths x bounces)", "value": v, "unit": "Msamples/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "steps_executed": len(vals), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, bounded=None if same else f"CPU arm runs a bounded sample of it: {w}x{h}, {budget} spp"),
        "cpu_baseline": cb, "e2e": {"value": v, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    ref = converged_reference(args.scene, w, h) if same else None
    if ref is not None:
        line["relmse"] = {"reference_algorithm": relmse(vals[-1]["image"], ref), "spp": budget, "against": f"scenes/ref/{args.scene}_{w}x{h}_ref.npy"}
    emit_line(line)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"film": vals[-1]["image"]})


# ------------------------------------------------------------------------------------------- GPU arm

def gpu_arm(args):
    import torch
    from ppg_b200 import capi
    from ppg_b200.integrator import GuidedPathTracer, torch_allreduce
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist      # rendezvous + bootstrap of the library's own NCCL communicator + the max-over-ranks of the timings
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    sc = load_scene(args.scene, args.width, args.height)
    props = scene_props(args, sc)
    g = GuidedPathTracer(props, device=local)
    g.set_scene(sc)
    comm = "single rank"
    if world > 1:
        if args.comm == "nccl":
            g.init_nccl(); comm = "ncclAllReduce enqueued on the render stream by libppg_b200.so (ppg_nccl_init)"
        else:
            g.set_shard(rank, world); g.set_allreduce(torch_allreduce()); comm = "torch.distributed.all_reduce through the ppg_set_allreduce callback"

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- `value`: inputs resident in HBM, film left in HBM
    try:
        uuid = str(torch.cuda.get_device_properties(local).uuid)
    except Exception:
        uuid = None
    sampler = ClockSampler(local, uuid); sampler.start()
    for _ in range(args.warmup):
        g.render_device()
    barrier()
    sampler.region(True)
    t0 = time.perf_counter()
    stats = []
    film_ptr = None
    for _ in range(args.steps):
        film_ptr, st = g.render_device()
        stats.append(st)
    barrier()
    wall = time.perf_counter() - t0
    sampler.region(False)
    film = device_film(film_ptr, args.height, args.width) if args.dump_outputs and rank == 0 else None     # before the e2e steps reuse the film buffer
    dev_ms = sum(s["render_device_ms"] for s in stats)          # CUDA events on the library's launching stream
    verts = sum(s["total_vertices"] for s in stats); paths = sum(s["total_paths"] for s in stats)
    launches = sum(s["kernel_launches"] for s in stats)
    if dist is not None:
        t = torch.tensor([dev_ms, wall * 1e3], device="cuda", dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, wall_ms = float(t[0]), float(t[1])
        c = torch.tensor([verts, paths, launches], device="cuda", dtype=torch.float64); dist.all_reduce(c, op=dist.ReduceOp.SUM)
        verts, paths, launches = (int(x) for x in c.tolist())
    else:
        wall_ms = wall * 1e3
    value = verts / (dev_ms * 1e-3) / 1e6

    # ---- `e2e`: host buffers through the public call; scene upload (H2D) and film download (D2H) inside the timed region
    arrays = g._scene_arrays
    h2d = int(sum(getattr(arrays, n).nbytes for n in ("positions", "normals", "uvs", "indices", "triangle_shape", "shapes", "bsdfs", "radiance", "tables", "texels", "env_texels") if hasattr(arrays, n)))
    d2h = args.width * args.height * 3 * 4
    barrier()
    e2e_steps = max(1, min(args.steps, 3))
    sampler.region(True)
    t0 = time.perf_counter(); ev = 0; img = None
    for _ in range(e2e_steps):
        g.set_scene(sc)
        if world > 1 and args.comm != "nccl":
            g.set_shard(rank, world)
        img, st = g.render()
        ev += st["total_vertices"]
    barrier()
    e2e_wall = time.perf_counter() - t0
    clocks = sampler.stop()                                      # samples cover both timed regions (device-resident and end-to-end)
    if dist is not None:
        t = torch.tensor([e2e_wall], device="cuda", dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX); e2e_wall = float(t[0])
        c = torch.tensor([ev], device="cuda", dtype=torch.float64); dist.all_reduce(c, op=dist.ReduceOp.SUM); ev = int(c[0])
    e2e_value = ev / e2e_wall / 1e6

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (bounce: raygen/intersect/shade/guide/compact), SURVEY 8d
    peak, peak_src = peaks()
    train_v = sum(i["vertices"] for s in stats for i in s["iterations"] if not i["is_final"])
    final_v = sum(i["vertices"] for s in stats for i in s["iterations"] if i["is_final"])
    rec_w = [(i["recorded_vertices"], i["s_tree_depth_avg"]) for s in stats for i in s["iterations"] if i["recorded_vertices"]]
    d_s = float(sum(n * d for n, d in rec_w) / max(1, sum(n for n, _ in rec_w))) if rec_w else 11.0
    dd = [i["depth_avg"] for s in stats for i in s["iterations"] if i["depth_avg"] > 0]
    d_d = float(np.mean(dd)) if dd else 5.5
    full_rec = any(k in props and props[k] not in ("none", "nearest") for k in ("bsdfSamplingFractionLoss", "spatialFilter"))
    b_bounce_train = 368 + (96 if full_rec else 0) + 16 * d_s + 24 * d_d        # path state 160 + hit record 32 + triangle 96 + vertex record write 80 (176 with the full record) + tree descents
    b_bounce_final = 288 + 16 * d_s + 24 * d_d
    bounce_ms = sum(s["kernel_ms"]["bounce"] for s in stats); bounce_n = sum(s["kernel_count"]["bounce"] for s in stats)
    my_train = sum(i["vertices"] for i in stats[0]["iterations"] if not i["is_final"]) * len(stats)   # rank 0's share when sharded
    my_final = sum(i["vertices"] for i in stats[0]["iterations"] if i["is_final"]) * len(stats)
    alg_bytes = my_train * b_bounce_train + my_final * b_bounce_final
    achieved = alg_bytes / (bounce_ms * 1e-3) / 1e9 if bounce_ms > 0 else 0.0
    traffic = None; traffic_src = None
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tp) and world == 1:           # measured with ncu at N = 1 for the default workload only; other shapes: null, not a borrowed constant
        try:
            tj = json.load(open(tp)); ent = tj.get(args.scene) if isinstance(tj.get(args.scene), dict) else (tj if args.scene == "cbox" else None)
            if ent and (ent.get("width", 1024), ent.get("budget", 252)) == (args.width, args.budget):
                traffic = ent.get("bounce_dram_bytes_per_launch"); traffic_src = ent.get("source")
        except Exception:
            traffic = None
    kname = "bounce_kernel (ray generation + intersection + shade + S/D-tree guide + compaction; one launch per path depth)"
    if args.scene != "cbox":
        kname += " + trace_kernel (nearest hits of wavefronts >= 32768 paths, persistent warps; timed together with the bounce launch it feeds)"
    roofline = {"bound": "hbm", "kernel": kname,
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_vertex": {"training": b_bounce_train, "final": b_bounce_final, "d_S": d_s, "d_D": d_d},
                "launches": int(bounce_n), "avg_launch_ms": bounce_ms / max(1, bounce_n),
                "kernel_ms_share": {k: sum(s["kernel_ms"][k] for s in stats) / max(1e-9, sum(s["render_device_ms"] for s in stats)) for k in capi.KERNEL_CLASSES},
                "pipeline_frac": (train_v * (468 + 16 * d_s + 48 * d_d) + final_v * (296 + 16 * d_s + 24 * d_d)) / (dev_ms * 1e-3) / 1e9 / peak / max(1, world),
                "what_actually_bounds_it": "issue / latency, not DRAM: the algorithmic bytes are mostly served by shared memory, L1 and the 126 MB L2 (measured DRAM traffic is `traffic`, "
                                           "a fraction of the algorithmic figure); see profiles/ for warp-issue utilisation and active lanes per instruction"}

    # ---- CPU baseline on the box's host cores (N = 1 only) and the metric's second half: equal-spp relMSE against a converged image
    cores = host_cores()
    cpu = None; rel = None
    ref = converged_reference(args.scene, args.width, args.height) if not args.budget_seconds else None
    if ref is not None and img is not None:
        rel = {"gpu": relmse(img, ref), "spp": args.budget, "against": f"scenes/ref/{args.scene}_{args.width}x{args.height}_ref.npy (the product at 32768 spp)"}
    if not args.no_cpu_baseline and world == 1:
        w, h, budget, same = cpu_sample_size(args)
        r = cpu_run(args, w, h, budget, cores)
        cpu = cpu_line_fields(r, cores, same)
        if rel is not None and same:
            rel["reference_algorithm"] = relmse(r["image"], ref)
            rel["gpu_over_reference"] = rel["gpu"] / rel["reference_algorithm"]
            rel["gpu_vs_reference_image"] = relmse(img, r["image"])
    line = {
        "metric": "Msamples/sec (paths x bounces)", "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args), "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "Msamples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps},
        "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "relmse": rel, "collective": comm,
        "wall_ms_per_step": wall_ms / args.steps, "kernel_ms_per_step": sum(sum(s["kernel_ms"].values()) for s in stats) / args.steps, "mpaths_per_s": paths / (dev_ms * 1e-3) / 1e6,
        "final_variance": stats[-1]["final_variance"], "iterations": stats[-1]["n_iterations"], "total_passes": stats[-1]["total_passes"],
        "sub_batches": stats[-1]["sub_batches"], "truncated_paths": stats[-1]["truncated_paths"], "dropped_records": stats[-1]["dropped_records"], "invalid_rays": stats[-1]["invalid_rays"],
    }
    if args.verbose:
        for it in stats[-1]["iterations"]:
            print({k: (round(v, 4) if isinstance(v, float) else v) for k, v in it.items() if k in ("iteration", "passes", "seconds", "reset_seconds", "build_seconds", "variance", "s_tree_leaves", "vertices", "nodes_avg", "depth_avg", "s_tree_depth_avg")}, file=sys.stderr)
        print({"render_device_ms": stats[-1]["render_device_ms"], "render_seconds": stats[-1]["render_seconds"], "kernel_ms": stats[-1]["kernel_ms"]}, file=sys.stderr)
    emit_line(line)
    if film is not None:
        dump_outputs(args.dump_outputs, {"film": film})
    if dist is not None:
        dist.destroy_process_group()


def device_film(ptr, h, w):
    """Host copy of the H x W x 3 float32 film that ppg_render_device left in HBM."""
    import torch

    class _Film:
        __cuda_array_interface__ = {"shape": (h, w, 3), "typestr": "<f4", "data": (ptr, False), "version": 3}
    torch.cuda.synchronize()
    return torch.as_tensor(_Film(), device="cuda").cpu().numpy().copy()


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: what the timed path returned in its last step, one DIR/<name>.npy per array (float32 / float64), so that two
    builds run with the same arguments (same scene, same seed) can be compared output for output.  A film larger than 64 MB is
    stored as a fixed, seeded sample of its pixels: DIR/<name>_sample.npy (N x 3) and the flat pixel indices DIR/<name>_sample_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        if a.nbytes <= DUMP_LIMIT:
            np.save(os.path.join(out_dir, name + ".npy"), a)
            continue
        px = a.reshape(-1, a.shape[-1])
        n = DUMP_LIMIT // 2 // px[0].nbytes
        idx = np.sort(np.random.default_rng(0).choice(len(px), n, replace=False))
        np.save(os.path.join(out_dir, name + "_sample.npy"), px[idx])
        np.save(os.path.join(out_dir, name + "_sample_index.npy"), idx.astype(np.float64))


_REAL_STDOUT = None


def quiet_stdout():
    """stdout carries exactly ONE JSON line: everything else a library prints there (NCCL's version banner, ...) is sent to stderr."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit_line(line):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        os.write(1, data)
    else:
        os.write(_REAL_STDOUT, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scene", default="cbox", choices=sorted(SCENES))
    ap.add_argument("--size", type=int, default=0, help="film width (height follows the scene's aspect); default: the BASELINE resolution")
    ap.add_argument("--budget", type=int, default=0, help="spp budget of one step (default per scene)")
    ap.add_argument("--budget-seconds", type=float, default=0.0, help="run the literal time-budget configuration instead")
    ap.add_argument("--comm", default="nccl", choices=["nccl", "torch"], help="N > 1: the library's own NCCL communicator (default) or the torch.distributed callback")
    ap.add_argument("--cpu-bounded", action="store_true", help="CBOX: time the CPU arm on the bounded 512^2 / 60 spp sample instead of the full configuration")
    ap.add_argument("--cpu-seconds", type=float, default=150.0, help="reference arm: stop repeating once this much time has been spent")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the film of the last timed step (H x W x 3 float32) as DIR/film.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    quiet_stdout()
    _, W, H, spp, _ = SCENES[args.scene]
    args.width = args.size or W
    args.height = (args.size * H // W) if args.size else H
    args.budget = args.budget or spp
    if args.impl == "reference":
        reference_arm(args)
    else:
        gpu_arm(args)


if __name__ == "__main__":
    main()
