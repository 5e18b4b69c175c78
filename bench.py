#!/usr/bin/env python3
"""
bench.py — headline benchmark of the B200 wavefront path tracer.

Metric (BASELINE.json): Mrays/s at 1920x1080, 8 bounces, 1 sample per pixel, where
  rays = sum_b N_ext[b] + sum_b N_shadow[b]   (rays actually submitted to BVH traversal, SURVEY 8d)
A "step" is one frame: Reset + Integrate with sample_idx = 0, so every step traces identical rays.

  python bench.py --gpus N --steps K --warmup W [--scene CornellBox] [--impl reference]

One process per GPU (torchrun for N > 1): the image is partitioned by scanline (row y -> rank y % N,
weak in nothing: total work fixed => "strong" scaling), each rank runs the whole wavefront on its rows,
and ONE gather of the radiance slabs to rank 0 belongs to every frame (inside the timed region): an NCCL gather after the frame, or —
above 4 ranks — the fused gather, in which the frame kernels store finished pixels into rank 0's buffer over NVLink peer memory.

The JSON line carries: value (HBM-resident, device-timed, max over ranks), e2e (through the public API with
host buffers: camera upload + frame + resolve + device->host image), roofline (dominant kernel, algorithmic
bytes / CUDA-event time vs MEASURED_PEAKS.json), cpu_baseline (the reference's own kernels compiled for the
CPU, oracle/_ref, or the oracle port), clocks sampled during the timed region, gpu_launches.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

WORKLOADS = {
    # name: (scene, width, height, max_bounces)
    "CornellBox": ("CornellBox", 1920, 1080, 8),          # BASELINE configs[1] — the headline
    "ShaderBalls": ("ShaderBalls", 1920, 1080, 8),        # configs[2]
    "CornellBox_Dragon": ("CornellBox_Dragon", 3840, 2160, 16),   # configs[3]
    "Synthetic10M": ("Synthetic10M", 1920, 1080, 8),      # configs[4]: 183 x ShaderBalls = 10 026 570 triangles
}


DUMP_LIMIT = 64_000_000                                    # --dump-outputs: bytes of all files together (.npy headers included)
DUMP_COUNTERS = ("n_ext", "n_miss", "n_emissive_hits", "n_shadow", "n_cont", "n_unoccluded")   # rows of frame_counters.npy


def dump_arrays(rad, counters):
    """The --dump-outputs files of a frame: radiance (h x w x 4 float32) and the per-bounce counters (float64).  When they
    would not fit DUMP_LIMIT, the radiance becomes a fixed, seeded sample of pixels (float32 RGBA) plus those pixels' indices
    (float64, exact): 24 bytes per sampled pixel, the sample sized so that every file fits with room for the .npy headers."""
    out = {"frame_counters": counters}
    if rad.nbytes + counters.nbytes + 4096 <= DUMP_LIMIT:
        out["radiance"] = rad
        return out
    flat = rad.reshape(-1, 4)
    n = (DUMP_LIMIT - counters.nbytes - 4096) // 24
    pix = np.sort(np.random.default_rng(0).choice(len(flat), n, replace=False))
    out["radiance_sample"], out["radiance_sample_pixels"] = flat[pix], pix.astype(np.float64)
    return out


def load_workload_scene(name, w, h, copies=183):
    """Scene arrays + camera of a workload.  Synthetic10M is generated (raytracing_b200/synthetic.py) and its BVH
    is built on the host by every rank (deterministic, so all ranks hold identical bytes)."""
    from raytracing_b200 import scene_io
    from raytracing_b200.camera import default_camera
    if name == "Synthetic10M":
        import pickle
        import tempfile
        from raytracing_b200 import synthetic
        # the scene (numpy replication + host BVH build, about a minute) is cached per box: several processes of one run reuse it
        cache = os.path.join(tempfile.gettempdir(), f"rt_b200_synthetic_{copies}_{w}x{h}.pkl")
        try:
            sc = pickle.load(open(cache, "rb"))
        except Exception:
            sc = synthetic.bistro_scale_scene(scene_io.load_scene("ShaderBalls"), copies, w, h)
            try:
                tmp = cache + f".{os.getpid()}"
                pickle.dump(sc, open(tmp, "wb"), protocol=4)
                os.replace(tmp, cache)
            except OSError:
                pass
        return sc, sc["camera_pose"]
    return scene_io.load_scene(name), default_camera(w, h)


def workload_string(name, w, h, mb):
    """config.workload — the same text in both arms (the driver compares the two strings)."""
    return f"{name} {w}x{h} 1spp {mb}-bounce, default camera of the workload, sample_idx 0, Reset+Integrate per step"


def algorithmic_bytes(st, mb, n_pix):
    """SURVEY 8(d): compulsory traffic of the reference layout, from per-bounce counters.
    Returns (total bytes per frame, bytes attributable to the fused extend+shade kernel)."""
    s = lambda k: st[k][: mb + 1].astype(np.float64)
    n_ext, n_miss, n_shadow, n_cont = s("n_ext"), s("n_miss"), s("n_shadow"), s("n_cont")
    n_hit = n_ext - n_miss
    n_unocc, n_emis = s("n_unoccluded"), s("n_emissive_hits")
    v_ext, t_ext, v_sh, t_sh = s("nodes_ext"), s("tris_ext"), s("nodes_shadow"), s("tris_shadow")
    raygen = 52.0 * n_pix
    trace = (48 * n_ext + 48 * (v_ext + t_ext)).sum()                                     # Ray in, Hit out, node + triangle fetches
    shade = (52 * n_miss + 264 * n_hit + 52 * n_shadow + 36 * n_cont + 32 * n_emis).sum() # miss + hit-surface streams
    shadow = (36 * n_shadow + 48 * (v_sh + t_sh) + 4 * n_shadow + 52 * n_unocc).sum()     # any-hit trace + accumulate
    return raygen + trace + shade + shadow, trace, shade, shadow


class ClockSampler(threading.Thread):
    """SM clock, power and throttle reasons sampled through NVML every ~2 ms DURING the timed region
    (same quantities as the nvidia-smi line of B200_PROFILING.md; nvidia-smi itself is too slow for a ~40 ms region)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.sm, self.power, self.reason_bits, self.stop_flag, self.err = index, [], [], 0, False, None
        self.sm_max = None
        self.nv = self.h = None

    def prepare(self):
        """NVML start-up (tens of ms) happens here, before the timed region, so that even a 10 ms region is sampled."""
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.index]) if vis and vis.split(",")[0].isdigit() else self.index
            self.nv, self.h = nv, nv.nvmlDeviceGetHandleByIndex(idx)
            self.sm_max = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
        except Exception as e:           # noqa: BLE001
            self.err = repr(e)
        return self

    def sample(self):
        nv, h = self.nv, self.h
        self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
        try:
            self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
        except Exception:
            pass
        self.reason_bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))

    def run(self):
        if self.err is not None:
            return
        try:
            while not self.stop_flag:
                self.sample()
                time.sleep(0.001)
        except Exception as e:           # noqa: BLE001
            self.err = repr(e)

    def summary(self):
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": ["nvml unavailable: %s" % self.err]}
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.sm_max, "reasons": [n for b, n in names.items() if self.reason_bits & b],
                "samples": len(sm), "power_w_max": max(self.power) if self.power else None}


def measured_peak_hbm():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def issue_roofline(name, world, ktimes, steps, sm_mhz, n_sms, peak_hbm, alg_of):
    """Roofline of the step's dominant kernel class from MEASURED quantities: CUDA-event time of this run (ktimes) and the
    per-frame instruction / DRAM counters of the committed ncu capture of the same workload (profiles/traffic.json, written
    by profiles/make_summaries.py from `ncu --set full`).  Two ceilings are evaluated and the binding one is reported:
      issue: warp instructions per second / (SMs x 4 schedulers x SM clock)   [one warp instruction per scheduler and clock]
      hbm:   DRAM bytes per second / MEASURED_PEAKS.json hbm_gbs
    plus the lane occupancy (thread instructions / 32 x warp instructions): the share of the issued lanes that did work."""
    try:
        tj = json.load(open(os.path.join(REPO, "profiles", "traffic.json")))
        wk = tj["workloads"][name]["kernels"]
        tag = tj["workloads"][name].get("tag")
    except Exception:
        wk, tag = {}, None
    issue_peak = n_sms * 4 * sm_mhz * 1e6                      # warp instructions per second
    rows = {}
    for k, (ms, n) in ktimes.items():
        if not n or ms <= 0 or k not in alg_of:
            continue
        sec = ms * 1e-3 / steps                                # seconds per frame spent in this kernel class
        row = {"kernel": k, "ms_per_step": ms / steps, "launches_per_step": n / steps,
               "algorithmic_GBs": alg_of[k] / world / sec / 1e9}
        c = wk.get(k)
        if c:
            scale = 1.0 / world                                # counters were captured on the whole frame; a rank owns 1/world of it
            inst, tinst, dram = c["inst_per_frame"] * scale, c["thread_inst_per_frame"] * scale, c["dram_bytes_per_frame"] * scale
            row.update({"issue_achieved_Ginst_s": inst / sec / 1e9, "issue_frac": inst / sec / issue_peak,
                        "lane_occupancy": tinst / (32.0 * inst), "hbm_achieved_GBs": dram / sec / 1e9, "hbm_frac": dram / sec / 1e9 / peak_hbm,
                        "traffic_bytes_per_launch": dram / max(n / steps, 1), "warp_inst_per_frame": inst,
                        "ncu_issue_active_pct": c.get("issue_active_pct"), "ncu_warps_active_pct": c.get("warps_active_pct")})
        rows[k] = row
    if not rows:
        return {"bound": None, "frac": None, "note": "no per-kernel times"}
    dom = max(rows, key=lambda k: rows[k]["ms_per_step"])
    d = rows[dom]
    out = {"kernel": dom, "kernel_ms_per_step": d["ms_per_step"], "kernel_launches_per_step": d["launches_per_step"],
           "peak_issue_Ginst_s": issue_peak / 1e9, "sm_mhz_used": sm_mhz, "n_sms": n_sms, "counter_source": f"profiles/traffic.json ({tag})" if tag else None,
           "other_kernels": [v for k, v in rows.items() if k != dom]}
    if "issue_frac" in d:
        issue_bound = d["issue_frac"] >= d["hbm_frac"]
        # neither ceiling within a factor of two: the kernel waits — dependent L2/HBM fetches of the traversal and, for scenes with
        # a long tail of ray lengths, resident warps that have run out of work while the slowest rays finish (ncu: warps active)
        label = ("issue" if issue_bound else "hbm") if max(d["issue_frac"], d["hbm_frac"]) >= 0.5 else "latency"
        out.update({"bound": label, "ncu_warps_active_pct": d.get("ncu_warps_active_pct"), "ncu_issue_active_pct": d.get("ncu_issue_active_pct"),
                    "achieved": d["issue_achieved_Ginst_s"] if issue_bound else d["hbm_achieved_GBs"],
                    "peak": issue_peak / 1e9 if issue_bound else peak_hbm,
                    "unit": "Gwarp-inst/s" if issue_bound else "GB/s",
                    "frac": d["issue_frac"] if issue_bound else d["hbm_frac"],
                    "issue": {"achieved": d["issue_achieved_Ginst_s"], "peak": issue_peak / 1e9, "unit": "Gwarp-inst/s", "frac": d["issue_frac"],
                              "lane_occupancy": d["lane_occupancy"], "effective_frac": d["issue_frac"] * d["lane_occupancy"]},
                    "hbm": {"achieved": d["hbm_achieved_GBs"], "peak": peak_hbm, "unit": "GB/s", "frac": d["hbm_frac"]},
                    "traffic": d["traffic_bytes_per_launch"]})
    else:
        out.update({"bound": None, "achieved": None, "peak": None, "unit": None, "frac": None, "traffic": None,
                    "note": f"no committed ncu counters for workload {name} in profiles/traffic.json"})
    out["algorithmic"] = {"achieved_GBs": d["algorithmic_GBs"], "note": "SURVEY 8(d) byte model (48 B per BVH node visit / triangle test); "
                          "secondary figure, not a bound: node and triangle fetches are L1/L2 hits"}
    return out


def host_threads() -> int:
    """Threads the CPU arm may really use: the affinity mask, capped by the cgroup CPU quota when one is set."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(np.ceil(int(quota) / int(period)))))
    except (OSError, ValueError):
        pass
    return max(1, n)


def cpu_reference_frame(scene, cam, w, h, mb, budget_s, threads):
    """Times the reference's CPU implementation of the path (oracle/_ref if built, else the oracle port) on a bounded
    sample: rows y % step == 0 of the same frame.  Returns (Mrays/s, kind, cores, sample description, seconds)."""
    os.environ["OMP_NUM_THREADS"] = str(threads)
    os.environ.setdefault("OMP_WAIT_POLICY", "passive")        # shared boxes: idle workers sleep instead of spinning
    from oracle import refbind
    from oracle.orcbind import Oracle
    use_ref = refbind.available()
    o = Oracle(scene)
    # probe on a sparse sample to size the bounded one (the port and _ref are bit-identical; the port is the cheaper probe)
    t0 = time.perf_counter()
    _, _, st = o.render(cam, w, h, mb, row_first=0, row_step=64, want_hits=False)
    probe = time.perf_counter() - t0
    est_full = probe * 64 * (4.0 if use_ref else 1.0)
    step = max(1, int(np.ceil(est_full / budget_s)))
    if use_ref:
        r = refbind.RefRenderer().open_arrays(scene)
        r.begin(w, h); r.set_camera(cam); r.set_max_bounces(mb)
        r.set_row_sample(0, step)
        t0 = time.perf_counter(); r.integrate(); dt = time.perf_counter() - t0
        s = r.stats()
        rays = float(s["n_ext"][: mb + 1].sum() + s["n_shadow"][: mb + 1].sum())
        r.close()
        kind = "reference"
    else:
        t0 = time.perf_counter()
        _, _, st = o.render(cam, w, h, mb, row_first=0, row_step=step, want_hits=False)
        dt = time.perf_counter() - t0
        rays = float(st["n_ext"][: mb + 1].sum() + st["n_shadow"][: mb + 1].sum())
        kind = "port"
    rows = len(range(0, h, step))
    sample = f"rows y%{step}==0 of the {w}x{h}x{mb}-bounce frame ({rows} rows, {rays / 1e6:.2f} Mrays), OpenMP over work-items"
    return rays / dt / 1e6, kind, threads, sample, dt


def run_reference_arm(args, workload):
    """--impl reference: the reference's own CPU implementation of the path on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name, w, h, mb = workload
    scene, cam = load_workload_scene(name, w, h, args.copies)
    cores = host_threads()
    total_budget = args.cpu_budget
    per_step = max(2.0, total_budget / (args.steps + args.warmup))
    vals, info = [], None
    for i in range(args.warmup + args.steps):
        v, kind, c, sample, dt = cpu_reference_frame(scene, cam, w, h, mb, per_step, cores)
        if i >= args.warmup:
            vals.append((v, dt))
        info = (kind, c, sample)
    value = float(np.mean([v for v, _ in vals]))
    ms = float(np.mean([dt for _, dt in vals]) * 1e3)
    line = {
        "impl": "reference", "metric": "Mrays/sec @1920x1080x8-bounce", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(name, w, h, mb), "device": "host CPU"},
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": info[1], "kind": info[0], "sample": info[2]},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scene", default="CornellBox", choices=sorted(WORKLOADS))
    ap.add_argument("--stepwise", action="store_true", help="time the one-kernel-per-reference-step schedule instead of the fused one")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--gather", default="auto", choices=["auto", "fused", "nccl"],
                    help="N > 1: the frame's one collective — fused: the frame kernels push finished pixels into rank 0's buffer over NVLink peer memory "
                         "(falls back to nccl when the CUDA IPC mapping cannot be set up); nccl: one NCCL gather after the frame; auto (default): fused for "
                         "more than 4 ranks, where it was measured faster (8 GPUs: 0.380 vs 0.411 ms per frame; 4: 0.682 vs 0.671; 2: 1.238 vs 1.211)")
    ap.add_argument("--no-host-e2e", action="store_true", help="skip the end-to-end leg through the C++ host classes (librt_host.so)")
    ap.add_argument("--cpu-budget", type=float, default=150.0, help="--impl reference: seconds of CPU work for the whole run (split over warm-up + steps)")
    ap.add_argument("--traversal", type=int, default=None, help="RT_OPT_TRAVERSAL override (0 literal reference-order traversal, 1 child-box layout)")
    ap.add_argument("--frame-kernel", type=int, default=2, help="RT_OPT_FRAME_KERNEL: 2 by partition size (default), 1 one persistent kernel per frame, 0 one kernel per phase")
    ap.add_argument("--secondary", default="Synthetic10M", help="second north_star scene measured (device-timed, same N) and reported under 'secondary'; 'none' to skip")
    ap.add_argument("--secondary-steps", type=int, default=8)
    ap.add_argument("--no-graph", action="store_true", help="RT_OPT_GRAPH=0: launch every kernel of the frame individually")
    ap.add_argument("--no-pdl", action="store_true", help="RT_OPT_PDL=0: no programmatic dependent launch between the kernels of a frame")
    ap.add_argument("--overlap", type=int, default=2, help="RT_OPT_OVERLAP: 2 shadow pass inside the next traversal kernel (default), 1 second stream, 0 none")
    ap.add_argument("--no-overlap", action="store_true", help="RT_OPT_OVERLAP=0: shadow pass on the render stream (no concurrency with the next traversal)")
    ap.add_argument("--no-smem-bvh", action="store_true", help="RT_OPT_SMEM_BVH=0: fetch BVH records through L1 even for small scenes")
    ap.add_argument("--copies", type=int, default=183, help="Synthetic10M: number of ShaderBalls copies (183 = 10 026 570 triangles)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (radiance, per-bounce ray counters) to DIR/<name>.npy, "
                         "at most 64 MB in all; DIR is created if missing and is best kept outside the source tree")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; --impl reference does not run it")
    workload = WORKLOADS[args.scene]
    if args.impl == "reference":
        run_reference_arm(args, workload)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    from raytracing_b200 import capi

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the render path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # NCCL logs to stdout by default; stdout carries ONE JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import types

    def device_run(workload, n_steps):
        """Scene upload, one counter frame, warm-up, n_steps device-timed frames (CUDA events on the context's stream, barrier +
        synchronize on both sides, max over ranks), then the same frames once more with per-launch events for the per-kernel
        split.  Returns everything the JSON line and the end-to-end legs need."""
        name, w, h, mb = workload
        steps = n_steps
        scene, cam = load_workload_scene(name, w, h, args.copies)
        ctx = capi.Context(w, h, device=local_rank, rank=rank, world=world)
        if args.traversal is not None:
            ctx.set_option(capi.OPT_TRAVERSAL, args.traversal)
        ctx.upload_scene(scene)
        ctx.set_camera(cam)
        ctx.set_option(capi.OPT_FRAME_KERNEL, args.frame_kernel)
        if args.no_graph:
            ctx.set_option(capi.OPT_GRAPH, 0)
        ctx.set_option(capi.OPT_OVERLAP, 0 if args.no_overlap else args.overlap)
        if args.no_pdl:
            ctx.set_option(capi.OPT_PDL, 0)
        if args.no_smem_bvh:
            ctx.set_option(capi.OPT_SMEM_BVH, 0)
        stream = torch.cuda.ExternalStream(ctx.stream_handle(), device=torch.device("cuda", local_rank))

        # the local radiance slab as a torch tensor (zero copy) for the NCCL gather
        ptr, nbytes = ctx.radiance_device_ptr()
        n_local = ctx.local_pixel_count()

        class _Slab:
            __cuda_array_interface__ = {"shape": (n_local, 4), "typestr": "<f4", "data": (ptr, False), "version": 3, "strides": None}
        slab = torch.as_tensor(_Slab(), device=torch.device("cuda", local_rank))
        from raytracing_b200.distributed import FusedGather, RadianceGather
        gather = RadianceGather(w, h, rank, world, slab.device)
        fused = None
        if world > 1 and (args.gather == "fused" or (args.gather == "auto" and world > 4)) and not args.stepwise:
            fused = FusedGather(ctx, rank, world)
            if not fused.ok:
                if rank == 0:
                    print(f"[bench] fused gather unavailable ({fused.errors[0]}): NCCL gather instead", file=sys.stderr)
                fused = None

        def frame():
            ctx.reset()
            if args.stepwise:
                ctx.integrate_stepwise(mb)
            else:
                ctx.integrate(mb)                               # fused gather: delivers the pixels to rank 0 while it renders, then sets this rank's flag
            if world > 1:
                if fused is not None:
                    fused.wait()                                # rank 0's stream waits for every rank's flag: the frame is gathered
                else:
                    with torch.cuda.stream(stream):
                        gather.gather(slab)                     # the ONE collective of the frame (NCCL, NVLink/NVSwitch)

        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        # ---- one instrumented frame (untimed): per-bounce counters incl. traversal work -> rays/frame, algorithmic bytes
        ctx.set_option(capi.OPT_COUNT_TRAVERSAL, 1)
        ctx.reset(); ctx.integrate(mb); ctx.sync()
        st = ctx.frame_stats()
        ctx.set_option(capi.OPT_COUNT_TRAVERSAL, 0)
        counters = torch.tensor([float(st[k][: mb + 1].sum()) for k in ("n_ext", "n_shadow")] +
                                list(algorithmic_bytes(st, mb, n_local)), dtype=torch.float64, device=slab.device)
        if world > 1:
            dist.all_reduce(counters)
        rays_per_frame = float(counters[0] + counters[1])
        alg_total, alg_trace, alg_shade, alg_shadow = (float(counters[i]) for i in (2, 3, 4, 5))
        alg_of = {"trace_closest": alg_trace, "shade_queues": alg_shade, "shadow_accumulate": alg_shadow, "extend_shade": alg_trace + alg_shade,
                  "intersect": alg_trace, "hit": alg_shade, "intersect_shadow": alg_shadow}

        # ---- warm-up, then K timed steps: barrier + synchronize on both sides, CUDA events on the launching stream
        for _ in range(args.warmup):
            frame()
        barrier()
        launches0 = ctx.launch_count()
        sampler = ClockSampler(local_rank).prepare(); sampler.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record(stream)
        for _ in range(steps):
            frame()
        ev1.record(stream)
        if sampler.h is not None and sampler.err is None:
            try:
                sampler.sample()            # the K steps are enqueued and running: at least this sample is taken under load
            except Exception as e:          # noqa: BLE001
                sampler.err = repr(e)
        barrier()
        sampler.stop_flag = True
        ms_total = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=slab.device)
        if world > 1:
            dist.all_reduce(ms_total, op=dist.ReduceOp.MAX)
        ms_per_step = float(ms_total[0]) / steps
        launches = ctx.launch_count() - launches0
        sampler.join(timeout=2)
        if args.dump_outputs and workload == WORKLOADS[args.scene]:
            dump_outputs(args.dump_outputs, ctx, mb, slab.device)
        # Per-kernel durations for the roofline.  In the timed region above the frame is ONE CUDA-graph launch and the shadow
        # pass of a bounce runs inside the next bounce's traversal kernel, so per-launch CUDA events are neither possible (graph)
        # nor would they separate the two passes: the same K steps are run once more, in this same process, with
        # per-launch events on, individual launches and the overlap off.
        ctx.set_option(capi.OPT_KERNEL_TIMING, 1)
        ctx.set_option(capi.OPT_OVERLAP, 0)
        for _ in range(2):
            frame()
        barrier()
        ctx.kernel_times()
        for _ in range(steps):
            frame()
        barrier()
        ktimes = ctx.kernel_times()
        ctx.set_option(capi.OPT_KERNEL_TIMING, 0)
        if not args.no_overlap:
            ctx.set_option(capi.OPT_OVERLAP, args.overlap)
        value = rays_per_frame / (ms_per_step * 1e-3) / 1e6
        n_prim = torch.tensor([float(st["n_ext"][0]), float(st["n_miss"][0])], dtype=torch.float64, device=slab.device)
        if world > 1:
            dist.all_reduce(n_prim)
        primary_hit_fraction = 1.0 - float(n_prim[1]) / max(float(n_prim[0]), 1.0)
        # the collective alone, as its own operation (the NCCL gather of the radiance slabs to rank 0), device-timed on the render
        # stream, max over ranks — for the fused gather this is the cost that the frame kernels absorb
        collective_kind = None if world == 1 else ("fused into the frame kernel: finished pixels are stored into rank 0's buffer over NVLink peer memory "
                                                   "(CUDA IPC mapping), one completion flag per rank" if fused is not None else "one NCCL gather after the frame")
        collective_ms = None
        if world > 1:
            for _ in range(2):                          # the first NCCL gather of a process sets the communicator up
                with torch.cuda.stream(stream):
                    gather.gather(slab)
            barrier()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record(stream)
            for _ in range(steps):
                with torch.cuda.stream(stream):
                    gather.gather(slab)
            c1.record(stream)
            barrier()
            cm = torch.tensor([c0.elapsed_time(c1) / steps], dtype=torch.float64, device=slab.device)
            dist.all_reduce(cm, op=dist.ReduceOp.MAX)
            collective_ms = float(cm[0])
        n_sms = torch.cuda.get_device_properties(local_rank).multi_processor_count
        fk_used = args.frame_kernel == 1 or (args.frame_kernel == 2 and n_local <= n_sms * 7168)
        schedule = ("stepwise: one kernel per reference kernel" if args.stepwise else
                    ("one persistent kernel per frame, CTA-private wavefronts: T(b) [closest-hit trace(b) + shadow pass(b-1)] -> S(b) [shade hit/miss queues]" if fk_used else
                     "per-phase kernels: [closest-hit trace(b) + shadow pass(b-1)] -> hit/miss queues -> shade(b), one CUDA graph per frame"))

        return types.SimpleNamespace(**{k: v for k, v in locals().items() if k not in ("workload",)})

    def dump_outputs(out_dir, ctx, mb, device):
        """What a caller of the timed path receives after its last step: the accumulated radiance (h x w x 4, rows of every
        rank) and the frame's per-bounce ray counters, written by rank 0 (dump_arrays)."""
        rad = torch.from_numpy(ctx.read_radiance()).to(device)          # other ranks' rows are zero here
        st = ctx.frame_stats()
        counters = torch.tensor(np.stack([st[k][: mb + 1].astype(np.float64) for k in DUMP_COUNTERS]), device=device)
        if world > 1:
            dist.reduce(rad, dst=0)
            dist.reduce(counters, dst=0)
        if rank != 0:
            return
        os.makedirs(out_dir, exist_ok=True)
        for k, v in dump_arrays(rad.cpu().numpy(), counters.cpu().numpy()).items():
            np.save(os.path.join(out_dir, k + ".npy"), v)

    def destroy_context(c):
        """Rank 0's context owns the fused-gather buffer that the other ranks have mapped through CUDA IPC: they unmap (destroy
        their context) first, rank 0 frees after the barrier."""
        if c is None:
            return
        if world > 1:
            if rank != 0:
                c.destroy()
            torch.cuda.synchronize(); dist.barrier()
            if rank == 0:
                c.destroy()
        else:
            c.destroy()

    R = device_run(workload, args.steps)
    name, w, h, mb = workload
    ctx, frame, barrier, gather, slab, stream, scene, cam = R.ctx, R.frame, R.barrier, R.gather, R.slab, R.stream, R.scene, R.cam
    rays_per_frame, ms_per_step, value, ktimes, alg_of, launches, sampler = R.rays_per_frame, R.ms_per_step, R.value, R.ktimes, R.alg_of, R.launches, R.sampler
    alg_total = R.alg_total

    # ---- end to end through the public API with HOST buffers: camera H2D, frame, gather, resolve, image D2H
    host_img = torch.zeros((h, w, 4), dtype=torch.float32).pin_memory()
    host_np = host_img.numpy()
    cam_host = np.ascontiguousarray(cam)

    # N > 1 has two presentation paths: "parallel" — every rank resolves and reads back ITS rows into one shared, page-locked
    # host image (N PCIe links), one barrier completes the frame; "gathered" — rank 0 resolves the NCCL-gathered frame and
    # reads the whole image back over its one link.  Both are measured; the parallel one is the headline when available.
    shared = None
    if world > 1:
        try:
            from raytracing_b200.distributed import SharedHostImage
            shared = SharedHostImage(w, h, rank, world)
        except Exception as e:                         # collectively consistent: raised on every rank or on none
            print(f"[bench] parallel read-back unavailable: {e}", file=sys.stderr)
            shared = None

    def e2e_frame(parallel=False):
        ctx.set_camera(cam_host)                       # per-frame input (render.cpp:188): 64 B host -> device (kernel parameter)
        frame()                                        # N > 1: includes the gather of the radiance slabs to rank 0 (NCCL or fused)
        if world == 1:
            ctx.resolve(host_np)                       # resolve + device->host of the image; blocks
        elif parallel:
            ctx.resolve(shared.image)                  # this rank's rows -> the shared host image; blocks on this rank's stream
            shared.complete()                          # one barrier: the image is whole on the host
        elif rank == 0:                                # rank 0 presents: resolve the WHOLE gathered frame + device->host; blocks
            if R.fused is not None:
                ctx.resolve_gathered(R.fused.ptr, R.fused.stride, host_np)
            else:
                ctx.resolve_gathered(gather.recv_ptr, gather.recv_stride_bytes, host_np)
        if world > 1 and not parallel and R.fused is not None:
            dist.barrier()                             # the peers may not push the next frame into the buffer rank 0 is still presenting
    e2e_steps = max(3, min(args.steps, 20))

    def time_e2e(parallel):
        for _ in range(3):
            e2e_frame(parallel)
        reps = []
        for _ in range(2):                             # host-side hiccups (this loop is paced by the CPU) are not the path: best of two repetitions
            barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                e2e_frame(parallel)
            barrier()
            reps.append((time.perf_counter() - t0) * 1e3 / e2e_steps)
        ms = torch.tensor([min(reps)], dtype=torch.float64, device=slab.device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms, reps

    e2e_ms, e2e_reps = time_e2e(False)
    e2e_gathered_ms = None
    if shared is not None:                             # N > 1: the figure above is the gathered path; the parallel path is the headline
        e2e_gathered_ms = float(e2e_ms[0])
        e2e_ms, e2e_reps = time_e2e(True)
    e2e_value = rays_per_frame / (float(e2e_ms[0]) * 1e-3) / 1e6

    # same end-to-end work with the read-back pipelined (rt_resolve_async): the D2H of frame i overlaps frame i+1
    host_imgs = [host_img, torch.zeros((h, w, 4), dtype=torch.float32).pin_memory()]
    host_nps = [t.numpy() for t in host_imgs]

    def e2e_frame_pipelined(i):
        ctx.set_camera(cam_host)
        frame()
        if world == 1:
            ctx.resolve_async(host_nps[i & 1])
        elif rank == 0:
            if R.fused is not None:
                ctx.resolve_gathered(R.fused.ptr, R.fused.stride, host_nps[i & 1], wait=False)
            else:
                ctx.resolve_gathered(gather.recv_ptr, gather.recv_stride_bytes, host_nps[i & 1], wait=False)
        if world > 1 and R.fused is not None:
            dist.barrier()
    for i in range(2):
        e2e_frame_pipelined(i)
    ctx.resolve_wait(); barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        e2e_frame_pipelined(i)
    ctx.resolve_wait(); barrier()
    e2e_pipe_ms = torch.tensor([(time.perf_counter() - t0) * 1e3 / e2e_steps], dtype=torch.float64, device=slab.device)
    if world > 1:
        dist.all_reduce(e2e_pipe_ms, op=dist.ReduceOp.MAX)
    e2e_pipe_value = rays_per_frame / (float(e2e_pipe_ms[0]) * 1e-3) / 1e6

    # ---- the same end-to-end step through the C++ drop-in: librt_host.so's Render::RenderFrame() (SetCameraData + RequestReset +
    # Integrate(), which ends with ResolveRadiance into Render's page-locked host image) on ALL N devices behind one
    # CUDAPathTraceIntegrator (rt_create_multi: fan-out, partition and read-back inside the library, ONE caller thread).
    # Rank 0 drives it; under torchrun the other ranks wait on the CPU (a key of the rendezvous store — an NCCL barrier would keep a
    # spinning kernel on their GPUs, which rank 0's kernels would have to time-slice with).
    host_e2e = None
    barrier()
    if rank == 0 and not args.no_host_e2e:
        try:
            from raytracing_b200 import hostapi
            hs = hostapi.scene_from_arrays(scene)
            hr = hostapi.HostRender.with_env_image(hs, w, h, scene["env"], scene["env_width"], scene["env_height"], list(range(world)), schedule="frame")
            hr.set_max_bounces(mb); hr.set_camera(cam)
            for _ in range(3):
                hr.request_reset(); hr.render_frame()
            reps = []
            for _ in range(2):
                t0 = time.perf_counter()
                for _ in range(e2e_steps):
                    hr.set_camera(cam)                  # per-frame input (render.cpp:188); marks the camera as changed -> RequestReset -> frame restarts
                    hr.render_frame()
                reps.append((time.perf_counter() - t0) * 1e3 / e2e_steps)
            hms = min(reps)
            host_e2e = {"value": rays_per_frame / (hms * 1e-3) / 1e6, "unit": "Mrays/s", "ms_per_step": hms, "repetitions_ms_per_step": [round(x, 4) for x in reps],
                        "devices": world, "h2d_bytes_per_step": 64 * world, "d2h_bytes_per_step": w * h * 16,
                        "api": "librt_host.so: rt_host::Render::RenderFrame() = CameraController data -> Integrator::SetCameraData, RequestReset, Integrator::Integrate() "
                               "(15 virtuals of CUDAPathTraceIntegrator, whole-frame schedule: one rt_integrate per frame) ending in ResolveRadiance() into the page-locked "
                               "host image; one thread, rt_create_multi over the N devices, parallel read-back; best of 2 repetitions"}
            hr.close(); hs.close()
        except Exception as e:          # noqa: BLE001
            host_e2e = {"value": None, "error": repr(e)[:300]}
    if world > 1:
        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            store.set("rt_b200_host_leg_done", "1")
        else:
            store.wait(["rt_b200_host_leg_done"])
    barrier()

    # ---- second north_star scene (BASELINE configs[4]): device-timed on the same N GPUs, reported under "secondary"
    secondary = None
    sec_name = args.secondary if args.secondary in WORKLOADS and args.secondary != args.scene else None
    if sec_name:
        destroy_context(ctx)                             # the primary context is finished: free its queues before the 3 GB scene
        ctx = None
        S = device_run(WORKLOADS[sec_name], args.secondary_steps)
        sclk = S.sampler.summary()
        if rank == 0:
            s_peak, _ = measured_peak_hbm()
            s_mhz = float(sclk.get("sm_mhz") or sclk.get("sm_max_mhz") or 1965.0)
            _, sw, sh, smb = WORKLOADS[sec_name]
            secondary = {"metric": "Mrays/sec @1920x1080x8-bounce", "value": S.value, "unit": "Mrays/s", "n_gpus": world, "steps": args.secondary_steps,
                         "ms_per_step": S.ms_per_step, "config": {"workload": workload_string(sec_name, sw, sh, smb), "triangles": int(len(S.scene["triangles"])),
                                                                  "bvh_depth": int(S.scene.get("bvh_depth", 0)), "schedule": S.schedule, "partition": f"scanline y%{world}",
                                                                  "rays_per_step": S.rays_per_frame, "primary_hit_fraction": S.primary_hit_fraction},
                         "collective_ms": S.collective_ms, "collective": {"kind": S.collective_kind, "nccl_gather_alone_ms": S.collective_ms}, "gpu_launches": int(S.launches),
                         "roofline": issue_roofline(sec_name, world, S.ktimes, args.secondary_steps, s_mhz, S.n_sms, s_peak, S.alg_of),
                         "kernel_ms_per_step": {k: v[0] / args.secondary_steps for k, v in S.ktimes.items() if v[1]}, "clocks": sclk}
        destroy_context(S.ctx)

    if rank == 0:
        peak, peak_src = measured_peak_hbm()
        clk = sampler.summary()
        sm_mhz = float(clk.get("sm_mhz") or clk.get("sm_max_mhz") or 1965.0)
        roof = issue_roofline(name, world, ktimes, args.steps, sm_mhz, R.n_sms, peak, alg_of)
        roof["peak_source"] = peak_src
        roof["algorithmic_bytes_per_step"] = alg_total
        roof["whole_frame_algorithmic_GBs"] = alg_total / (ms_per_step * 1e-3) / 1e9
        roof["how"] = ("kernel time: CUDA events of THIS run (per-launch, per-phase kernels, shadow pass as its own kernel); instruction and DRAM "
                       "counters: committed ncu --set full capture of the same workload and kernels (profiles/); issue peak = SMs x 4 x SM clock")
        line = {
            "metric": "Mrays/sec @1920x1080x8-bounce", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(name, w, h, mb), "triangles": int(len(scene['triangles'])),
                       "schedule": R.schedule, "partition": f"scanline y%{world}",
                       "rays_per_step": rays_per_frame, "primary_hit_fraction": R.primary_hit_fraction,
                       "l2": "per-step working set (ray/shadow queues + radiance, ~365 MB at 1080p) exceeds the 126 MB L2; no explicit flush"},
            "e2e": {"value": e2e_value, "unit": "Mrays/s", "ms_per_step": float(e2e_ms[0]), "steps": e2e_steps,
                    "repetitions_ms_per_step": [round(x, 4) for x in e2e_reps], "h2d_bytes_per_step": 64,
                    "d2h_bytes_per_step": w * h * 16,          # the whole image reaches the host every step (N > 1: split over the ranks' links)
                    "api": ("rt_set_camera + rt_reset + rt_integrate + rt_resolve(host image), blocking per frame like ResolveRadiance/Finish(); best of 2 repetitions" if world == 1 else
                            (f"every rank: rt_set_camera + rt_reset + rt_integrate + gather to rank 0 [{'fused' if R.fused is not None else 'NCCL'}] + rt_resolve of its rows into ONE shared page-locked host "
                             "image (N PCIe links) + barrier; blocking per frame" if shared is not None else
                             f"every rank: rt_set_camera + rt_reset + rt_integrate + gather to rank 0 [{'fused' if R.fused is not None else 'NCCL'}]; rank 0: rt_resolve_gathered(whole host image), blocking per frame")),
                    "gathered_value": (rays_per_frame / (e2e_gathered_ms * 1e-3) / 1e6) if e2e_gathered_ms else None,
                    "gathered_api": "rank 0: rt_resolve_gathered(whole host image) after the gather (one PCIe link)" if e2e_gathered_ms else None,
                    "host_image_page_locked": (shared.pinned if shared is not None else True),
                    "pipelined_value": e2e_pipe_value, "pipelined_ms_per_step": float(e2e_pipe_ms[0]),
                    "pipelined_api": "same, with rt_resolve_async: image D2H of frame i overlaps frame i+1",
                    "host_cpp": host_e2e},
            "gpu_launches": int(launches),
            "roofline": roof,
            "collective_ms": R.collective_ms, "collective": {"kind": R.collective_kind, "nccl_gather_alone_ms": R.collective_ms},
            "kernel_ms_per_step": {k: v[0] / args.steps for k, v in ktimes.items() if v[1]},
            "kernel_timing_note": "kernel_ms_per_step: CUDA events per launch over K extra steps of this run with individual launches and the "
                                  "shadow pass as its own kernel (in the timed region the frame is one CUDA-graph launch in which the shadow pass of "
                                  "bounce b runs inside the traversal kernel of bounce b+1)",
            "clocks": clk,
        }
        if secondary is not None:
            line["secondary"] = secondary
        if not args.no_cpu_baseline and world == 1:
            # The CPU leg runs in a fresh process (the --impl reference arm, one bounded sample): this process has torch's OpenMP
            # runtime loaded and already configured, which would decide the thread count and wait policy for the oracle too.
            env = {k: v for k, v in os.environ.items() if k not in ("OMP_NUM_THREADS", "RANK", "LOCAL_RANK", "WORLD_SIZE")}
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "1",
                                  "--scene", args.scene, "--copies", str(args.copies), "--cpu-budget", "30"],
                                 capture_output=True, text=True, env=env, timeout=900)
            try:
                line["cpu_baseline"] = json.loads(out.stdout.strip().splitlines()[-1])["cpu_baseline"]
            except Exception:
                line["cpu_baseline"] = {"value": None, "unit": "Mrays/s", "error": (out.stderr or out.stdout)[-300:]}
        print(json.dumps(line))
    if shared is not None:
        shared.close()
    destroy_context(ctx)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
