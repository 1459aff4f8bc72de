#!/usr/bin/env python
"""bench.py -- headline benchmark of the resample hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl ours|reference] [--dump-outputs DIR]
  (N > 1: launched by torch.distributed.run, one rank per GPU; images are independent, so every rank
   resamples its own full batch -- weak scaling, no data-path collective.)

A "step" is one pass of the hot path over one batch of synthetic BGRA frames that are already resident
in HBM (`value`), and -- for `e2e` -- the same call sequence through the drop-in C ABI with HOST buffers,
host<->device copies inside the timed region.  `--impl reference` times the CPU oracle (a restatement of
the reference's algorithm; the Rust reference itself cannot be built offline) on the box's host cores.
Rank 0 prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json metric line: "Mpixels/sec (4K->512 Robidoux batch)"; configs[1] shape with the metric's filter
    "c2_4k_to_512_robidoux": dict(in_wh=(3840, 2160), out_wh=(512, 512), filter=2, batch=1024, alpha=0, compose=0, sharpen=0.0, cm=None),
    # configs[1] verbatim (Lanczos3)
    "c2_4k_to_512_lanczos3": dict(in_wh=(3840, 2160), out_wh=(512, 512), filter=6, batch=1024, alpha=0, compose=0, sharpen=0.0, cm=None),
    # configs[2]: 8K -> 1080p Robidoux, linear-light round trip, sharpen_percent=50 (the reference's only sharpening)
    "c3_8k_to_1080p_robidoux_sharpen": dict(in_wh=(7680, 4320), out_wh=(1920, 1080), filter=2, batch=256, alpha=0, compose=0, sharpen=50.0, cm=None),
    # configs[3]: 1080p -> 4K Mitchell upscale, sepia colour matrix, composited over an existing canvas
    "c4_1080p_to_4k_mitchell_sepia_over": dict(in_wh=(1920, 1080), out_wh=(3840, 2160), filter=14, batch=512, alpha=1, compose=1, sharpen=0.0, cm=0),
}
DEFAULT_WORKLOAD = "c2_4k_to_512_robidoux"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="override images per GPU per step")
    ap.add_argument("--alpha", type=int, default=-1, help="override alpha_meaningful (0/1)")
    ap.add_argument("--content", default="noise", choices=["noise", "gradient"])
    ap.add_argument("--e2e-images", type=int, default=48, help="host-buffer images per e2e step")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU-baseline sample time")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--no-others", action="store_true", help="skip the runs of the other BASELINE.json configurations")
    ap.add_argument("--ncu-traffic", action="store_true", help="measure the kernel's DRAM traffic with ncu and rewrite profiles/traffic_<workload>.json")
    ap.add_argument("--strip-cols", type=int, default=0, help="ring kernel: widest strip of output columns per warp (0 = library default)")
    ap.add_argument("--min-items", type=int, default=-1, help="ring kernel: band split target (-1 = library default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a fixed sample of the last step's output images to DIR/*.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.rows, self.proc, self.index, self.first = [], None, index, 0

    def mark(self):
        """samples taken from now on belong to the timed region"""
        self.first = len(self.rows)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for r in self.rows[max(0, self.first - 1):]:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def host_cpu_info() -> dict:
    """What the CPU arm can really use: the scheduler affinity AND the cgroup CPU quota (a container given 16 CPUs of a 128-thread
    host still sees 128 in sched_getaffinity), plus the CPU model.  `threads` is what the OpenMP runs are given."""
    try:
        aff = max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        aff = max(1, os.cpu_count() or 1)
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read().split()[0])
            break
        except Exception:
            continue
    model = None
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip(); break
    except Exception:
        pass
    eff = aff if quota is None else max(1, min(aff, int(quota + 0.999)))
    return {"threads": eff, "sched_affinity": aff, "cgroup_cpu_quota": quota, "cpu_model": model}


def host_threads() -> int:
    """host threads for the CPU arm (torchrun exports OMP_NUM_THREADS=1, so ask the scheduler and the cgroup instead)"""
    return host_cpu_info()["threads"]


def algorithmic_bytes_per_image(wl):
    iw, ih = wl["in_wh"]; ow, oh = wl["out_wh"]
    b = iw * ih * 4 + ow * oh * 4                    # SURVEY.md §8(d): read input once + write output once
    if wl["compose"] == 1:
        b += ow * oh * 4                             # + canvas read for compose-onto-canvas
    return b


# --------------------------------------------------------------------------------------------------
CPU_DISTINCT = 64       # distinct input frames the CPU arm cycles through (64 4K frames = 2.1 GB: far larger than any last-level cache)


class CpuArm:
    """The CPU oracle (OpenMP over images) on frames of the workload.  Inputs are generated once (C generator, same bytes as
    imageflow_b200.synth) and kept; a run of n images walks them cyclically, every job with its own canvas."""

    def __init__(self, wl, content, alpha, distinct):
        import oracle
        from imageflow_b200 import synth
        self.wl, self.alpha, self.oracle = wl, alpha, oracle
        iw, ih = wl["in_wh"]; ow, oh = wl["out_wh"]
        am = "mixed" if alpha else "opaque"
        self.ins = [oracle.synth_noise(iw, ih, seed=i, alpha_mode=am) if content == "noise" else synth.gradient_np(iw, ih) for i in range(distinct)]
        self.cv0 = [oracle.synth_noise(ow, oh, seed=100000 + i, alpha_mode="mixed") for i in range(distinct)] if wl["compose"] == 1 else None
        self.cm = oracle.color_filter_matrix(wl["cm"]) if wl["cm"] is not None else None

    def run(self, n_images, threads, keep_outputs=False):
        wl, oracle = self.wl, self.oracle
        ow, oh = wl["out_wh"]
        d = len(self.ins)
        outs = [self.cv0[i % d].copy() if self.cv0 is not None else np.zeros((oh, ow, 4), np.uint8) for i in range(n_images)]
        descs, keep = (oracle.Desc * n_images)(), []
        for i in range(n_images):
            descs[i] = oracle.make_desc(self.ins[i % d], outs[i], filter=wl["filter"], sharpen=wl["sharpen"], linear=True, alpha_meaningful=bool(self.alpha),
                                        compose=wl["compose"], color_matrix=self.cm, keep=keep)
        t0 = time.perf_counter()
        rc = oracle.lib().ifo_scale_and_render_batch(descs, n_images, threads)
        dt = time.perf_counter() - t0
        if rc:
            raise RuntimeError(f"oracle failed rc={rc}")
        return dt, (outs if keep_outputs else None)


def run_reference(args, wl, rank, world):
    """--impl reference: the CPU implementation of the path on the host cores (rank 0 only).  Every step is the workload's full
    batch (the same `config` as the GPU arm) unless that would take more than ~12 s per step on this host, then a bounded sample."""
    if rank != 0:
        return
    import oracle
    oracle.build()
    cpu = host_cpu_info()
    threads = cpu["threads"]
    alpha = wl["alpha"] if args.alpha < 0 else args.alpha
    iw, ih = wl["in_wh"]
    B = args.batch or wl["batch"]
    arm = CpuArm(wl, args.content, alpha, min(B, CPU_DISTINCT))
    arm.run(min(B, threads), threads)                                            # warm-up (tables, page faults)
    dt, _ = arm.run(min(B, 2 * threads), threads)
    per_image = dt / min(B, 2 * threads)
    n = B if per_image * B <= 12.0 else int(max(2 * threads, 12.0 / per_image))
    for _ in range(args.warmup):
        arm.run(n, threads)
    t = 0.0
    for _ in range(args.steps):
        d, _ = arm.run(n, threads)
        t += d
    mpx = n * args.steps * iw * ih / 1e6 / t
    sample = (f"{n} frames of {iw}x{ih} per step ({'the full batch' if n == B else f'bounded sample of the {B}-frame batch'}; {min(B, CPU_DISTINCT)} distinct frames, "
              f"cycled), OpenMP over images on {threads} threads")
    line = {"impl": "reference", "metric": "input Mpixels/s, " + args.workload, "value": mpx, "unit": "Mpx/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args, wl, alpha, n),
            "cpu_baseline": {"value": mpx, "unit": "Mpx/s", "cores": threads, "kind": "port", "sample": sample, "host": cpu},
            "e2e": {"value": mpx, "unit": "Mpx/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "CPU restatement of the reference algorithm (oracle/ifb_oracle.c); the Rust reference (zenresize) cannot be built offline"}
    print(json.dumps(line), flush=True)


def config_dict(args, wl, alpha, batch):
    iw, ih = wl["in_wh"]; ow, oh = wl["out_wh"]
    names = {2: "Robidoux", 6: "Lanczos", 14: "Mitchell"}
    return {"workload": args.workload, "in": f"{iw}x{ih}", "out": f"{ow}x{oh}", "filter": names.get(wl["filter"], str(wl["filter"])),
            "colorspace": "linear", "alpha_meaningful": bool(alpha), "compose": ["ReplaceSelf", "BlendWithSelf", "BlendWithMatte"][wl["compose"]],
            "sharpen_percent": wl["sharpen"], "color_matrix": "sepia" if wl["cm"] == 0 else None,
            "images_per_gpu_per_step": batch, "content": args.content, "parallelism": f"images sharded x{args.gpus}, no collective",
            "cache": "inputs (>= 8 GB per step) are far larger than the 126 MB L2; no explicit flush needed"}


# --------------------------------------------------------------------------------------------------
class DeviceWorkload:
    """One workload resident in HBM of one GPU: synthetic frames, canvases, the batch object and its descriptors."""

    def __init__(self, args, name, local, batch_override=0):
        import torch
        import imageflow_b200 as ifb
        from imageflow_b200 import synth
        self.torch, self.ifb, self.name = torch, ifb, name
        wl = self.wl = dict(WORKLOADS[name])
        dev = self.dev = torch.device("cuda", local)
        self.alpha = alpha = wl["alpha"] if args.alpha < 0 else args.alpha
        B = batch_override or args.batch or wl["batch"]
        iw, ih = wl["in_wh"]; ow, oh = wl["out_wh"]
        free, _total = torch.cuda.mem_get_info()
        per = iw * ih * 4 + 3 * ow * oh * 4
        if B * per > free * 0.9:
            B = max(1, int(free * 0.9 // per))
        self.B = B
        self.inp = torch.empty((B, ih, iw, 4), dtype=torch.uint8, device=dev)
        for i in range(B):
            if args.content == "noise":
                synth.noise_torch(iw, ih, seed=i, alpha_mode="mixed" if alpha else "opaque", device=dev, out=self.inp[i])
            else:
                synth.gradient_torch(iw, ih, device=dev, out=self.inp[i])
        self.canvas0 = None
        if wl["compose"] == 1:
            self.canvas0 = torch.empty((B, oh, ow, 4), dtype=torch.uint8, device=dev)
            for i in range(B):
                synth.noise_torch(ow, oh, seed=100000 + i, alpha_mode="mixed", device=dev, out=self.canvas0[i])
        self.out = torch.zeros((B, oh, ow, 4), dtype=torch.uint8, device=dev)
        self.cm = ifb.color_filter_matrix(wl["cm"]) if wl["cm"] is not None else None
        self.batch = ifb.Batch(local)
        if args.strip_cols:
            self.batch.set_option(ifb.Batch.OPT_STRIP_COLUMNS, args.strip_cols)
        if args.min_items >= 0:
            self.batch.set_option(ifb.Batch.OPT_MIN_ITEMS, args.min_items)
        self.params = ifb.ScaleAndRenderParams(w=ow, h=oh, sharpen_percent_goal=wl["sharpen"], interpolation_filter=ifb.Filter(wl["filter"]))
        jobs = [(ifb.BitmapWindow.from_torch(self.inp[i], alpha_meaningful=bool(alpha)),
                 ifb.BitmapWindow.from_torch(self.out[i], compose=ifb.BitmapCompositing(wl["compose"])), self.params, self.cm) for i in range(B)]
        self.descs, self.keep = self.batch.make_descs(jobs)
        self.stream = torch.cuda.current_stream().cuda_stream

    def step(self):
        if self.canvas0 is not None:
            self.out.copy_(self.canvas0)          # the composite reads the canvas: restore it so every step does identical work
        self.batch.enqueue(self.descs, self.stream)

    def warm(self, steps, seconds=0.5):
        t_w, n_w = time.perf_counter(), 0
        while n_w < max(steps, 3) or time.perf_counter() - t_w < seconds:     # >= 3 steps and >= 0.5 s: clocks ramp up
            self.step()
            n_w += 1
            if n_w % 8 == 0:
                self.torch.cuda.synchronize()

    def timed(self, steps):
        """`steps` timed steps; returns (total ms between the bracketing events, per-step kernel ms, host enqueue ms)"""
        torch = self.torch
        k_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        host_ms = []
        e0.record()
        for k in range(steps):
            if self.canvas0 is not None:
                self.out.copy_(self.canvas0)
            k_ev[k][0].record()
            t_h = time.perf_counter()
            self.batch.enqueue(self.descs, self.stream)
            host_ms.append((time.perf_counter() - t_h) * 1e3)
            k_ev[k][1].record()
        e1.record()
        return e0, e1, k_ev, host_ms

    def roofline(self, step_ms, host_ms):
        peak, peak_src = peaks()
        alg = algorithmic_bytes_per_image(self.wl) * self.B
        kern_ms = float(np.mean(step_ms))
        achieved = alg / (kern_ms / 1e3) / 1e9
        b = self.batch
        return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "peak_source": peak_src, "kernel_ms": kern_ms, "kernel_ms_min": float(np.min(step_ms)),
                "kernel_ms_all": [round(x, 4) for x in step_ms], "host_enqueue_ms": [round(x, 3) for x in host_ms], "algorithmic_bytes_per_launch": alg,
                "fused_jobs": b.fused_jobs, "generic_jobs": b.generic_jobs, "tile_jobs": b.tile_jobs}

    def check(self, content, n_chk=2):
        """parity spot check of the first frames against the oracle"""
        import oracle
        oracle.build()
        arm = CpuArm(self.wl, content, self.alpha, n_chk)
        _, outs = arm.run(n_chk, min(n_chk, os.cpu_count() or 1), keep_outputs=True)
        if self.canvas0 is not None:       # rerun once from the pristine canvas so that out holds exactly one composite
            self.out.copy_(self.canvas0)
            self.batch.enqueue(self.descs, self.stream)
        self.torch.cuda.synchronize()
        mx = 0
        for i in range(n_chk):
            mx = max(mx, int(np.abs(self.out[i].cpu().numpy().astype(np.int16) - outs[i].astype(np.int16)).max()))
        return {"images": n_chk, "max_abs_delta_vs_oracle": mx}

    def dump(self, out_dir, max_bytes=48 << 20):
        """Writes the batch's output images as a caller receives them: out.npy = float32 (rows, out_w, 4) BGRA rows, and
        out_rows.npy = float64 (rows, 2) of (image, row) for each.  All rows when they fit in `max_bytes`, else a seeded
        sample of rows that depends only on the batch geometry, so two builds run with the same arguments dump the same rows."""
        torch = self.torch
        B, oh, ow, _ = self.out.shape
        total = B * oh
        n = min(total, max_bytes // (ow * 4 * 4))
        rows = np.arange(total) if n == total else np.sort(np.random.default_rng(0).choice(total, n, replace=False))
        torch.cuda.synchronize()
        sel = self.out.reshape(total, ow, 4)[torch.from_numpy(rows).to(self.dev)]
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, "out.npy"), sel.to(torch.float32).cpu().numpy())
        np.save(os.path.join(out_dir, "out_rows.npy"), np.stack([rows // oh, rows % oh], axis=1).astype(np.float64))

    def close(self):
        self.batch.close()
        self.descs = self.keep = None
        del self.inp, self.out, self.canvas0
        self.torch.cuda.empty_cache()


def git_sha():
    try:
        return subprocess.run(["git", "rev-parse", "--short", "HEAD"], cwd=ROOT, capture_output=True, text=True).stdout.strip() or None
    except Exception:
        return None


def lib_digest():
    """identifies the build a traffic measurement belongs to: a digest of the library's SOURCES (the in-tree .so is rebuilt from
    them by __graft_entry__.build(); its bytes may differ between builds, what it is built from does not)"""
    import glob
    import hashlib
    h = hashlib.sha256()
    try:
        for f in sorted(glob.glob(os.path.join(ROOT, "imageflow_b200", "csrc", "*"))):
            if f.endswith((".cu", ".cuh", ".cc", ".h", ".inc", "Makefile")):
                h.update(os.path.basename(f).encode()); h.update(open(f, "rb").read())
        return h.hexdigest()[:16]
    except Exception:
        return None


def measure_traffic(args):
    """--ncu-traffic: one launch of the workload's kernel under ncu (dram bytes read + written), written to
    profiles/traffic_<workload>.json together with the kernel name and the digest of the library it was taken from."""
    import tempfile
    n = 64 if WORKLOADS[args.workload]["in_wh"][0] <= 3840 else 16
    csv_path = os.path.join(tempfile.mkdtemp(prefix="ifb200_ncu_"), f"traffic_{args.workload}.csv")
    cmd = ["ncu", "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum", "--clock-control", "none", "-k", "regex:hv_ring|fused_tile2|generic",
           "-s", "3", "-c", "1", "--csv", "--log-file", csv_path, sys.executable, os.path.abspath(__file__), "--workload", args.workload, "--batch", str(n),
           "--steps", "1", "--warmup", "3", "--no-cpu", "--no-e2e", "--no-check", "--no-others"]
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
    import csv
    rows = [row for row in csv.reader(open(csv_path)) if len(row) > 5]
    hdr = rows[0]
    name_i, metric_i, val_i, unit_i = hdr.index("Kernel Name"), hdr.index("Metric Name"), hdr.index("Metric Value"), hdr.index("Metric Unit")
    vals, kname = {}, None
    for row in rows[1:]:
        kname = row[name_i]
        v = float(row[val_i].replace(",", ""))
        u = row[unit_i].lower()
        mult = {"byte": 1, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}.get(u, 1)
        vals[row[metric_i]] = v * mult
    out = {"workload": args.workload, "kernel": kname, "images_per_launch": n, "dram_bytes_per_launch": vals["dram__bytes_read.sum"] + vals["dram__bytes_write.sum"],
           "dram_bytes_read": vals["dram__bytes_read.sum"], "dram_bytes_write": vals["dram__bytes_write.sum"], "git": git_sha(), "src_sha256_16": lib_digest(),
           "source": "bench.py --ncu-traffic: ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum --clock-control none, one launch after 3 warm-up launches"}
    json.dump(out, open(os.path.join(ROOT, "profiles", f"traffic_{args.workload}.json"), "w"), indent=1)
    print(json.dumps(out))


def main():
    args = parse()
    wl = dict(WORKLOADS[args.workload])
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, wl, rank, world)
        return
    if args.ncu_traffic:
        measure_traffic(args)
        return

    import torch
    import torch.distributed as dist
    import imageflow_b200 as ifb

    if not torch.cuda.is_available() or ifb.device_count() == 0:
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    iw, ih = wl["in_wh"]; ow, oh = wl["out_wh"]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    w = DeviceWorkload(args, args.workload, local)
    B, alpha = w.B, w.alpha
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()          # started before the warm-up so that nvidia-smi's start-up cost is not in the timed region
    w.warm(args.warmup)
    barrier()
    launches0 = w.batch.kernel_launches
    if rank == 0:
        sampler.mark()
    barrier()
    torch.cuda.cudart().cudaProfilerStart()      # `ncu --profile-from-start off` then lists the launches of the timed region only
    e0, e1, k_ev, host_ms = w.timed(args.steps)
    barrier()
    torch.cuda.cudart().cudaProfilerStop()
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        w.dump(args.dump_outputs)
    total_ms = e0.elapsed_time(e1)
    step_ms = [a.elapsed_time(b) for a, b in k_ev]
    launches = w.batch.kernel_launches - launches0
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    value = world * B * args.steps * iw * ih / 1e6 / (total_ms_max / 1e3)

    # ---- roofline of the dominant kernel (one launch per step)
    roofline = w.roofline(step_ms, host_ms)
    tfile = os.path.join(ROOT, "profiles", f"traffic_{args.workload}.json")
    if os.path.exists(tfile):
        try:
            tj = json.load(open(tfile))
            if tj.get("src_sha256_16") == lib_digest():      # only a measurement of a build of THESE sources describes this run
                roofline["traffic"] = tj["dram_bytes_per_launch"] * (B / tj["images_per_launch"])
                roofline["traffic_source"] = tj.get("source")
                roofline["traffic_kernel"] = tj.get("kernel")
            else:
                roofline["traffic_source"] = f"profiles/traffic_{args.workload}.json was measured on another build of the library (run bench.py --ncu-traffic)"
        except Exception:
            pass

    # ---- parity spot check against the oracle + CPU baseline (rank 0, N == 1 only for the baseline)
    check = None
    cpu_baseline = None
    if rank == 0 and not args.no_check:
        check = w.check(args.content)
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = host_cpu_info()
        threads = cpu["threads"]
        arm = CpuArm(wl, args.content, alpha, min(B, CPU_DISTINCT))
        arm.run(min(B, threads), threads)                                        # warm-up (tables, page faults)
        dt, _ = arm.run(min(B, 2 * threads), threads)
        n = int(max(2 * threads, min(B, round(args.cpu_seconds / max(dt, 1e-3) * min(B, 2 * threads)))))
        dt, _ = arm.run(n, threads)
        cpu_baseline = {"value": n * iw * ih / 1e6 / dt, "unit": "Mpx/s", "cores": threads, "kind": "port", "host": cpu,
                        "sample": f"{n} frames of {iw}x{ih} ({dt:.1f} s; {min(B, CPU_DISTINCT)} distinct frames, cycled), oracle/ifb_oracle.c OpenMP over images on {threads} threads"}
        del arm

    # ---- e2e: drop-in C ABI with HOST buffers, copies inside the timed region.  Headline = pinned buffers (what a caller that
    # cares would allocate); `pageable` = plain host memory, which is what imageflow's Bitmap gives the seam today
    # (aligned_buffer.rs:40-43).  Both are bound by the host link, not by the kernel.
    e2e = None
    if not args.no_e2e:
        ne = max(1, min(args.e2e_images, B))
        os.environ["IFB200_DEVICE"] = str(local)
        params, cm = w.params, w.cm

        def e2e_leg(pinned):
            h_in = torch.empty((ne, ih, iw, 4), dtype=torch.uint8)
            h_out = torch.zeros((ne, oh, ow, 4), dtype=torch.uint8)
            if pinned:
                h_in, h_out = h_in.pin_memory(), h_out.pin_memory()
            h_in.copy_(w.inp[:ne])
            h_cv0 = w.canvas0[:ne].cpu() if w.canvas0 is not None else None
            hjobs = [(ifb.BitmapWindow(h_in[i].data_ptr(), iw, ih, iw * 4, alpha_meaningful=bool(alpha)),
                      ifb.BitmapWindow(h_out[i].data_ptr(), ow, oh, ow * 4, compose=ifb.BitmapCompositing(wl["compose"])), params) for i in range(ne)]

            def e2e_step():
                if h_cv0 is not None:
                    h_out.copy_(h_cv0)
                ifb.scale_and_render_many([(wi, wc, p, cm) for (wi, wc, p) in hjobs])

            e2e_step()
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                e2e_step()
            barrier()
            dt = time.perf_counter() - t0
            tt = torch.tensor([dt], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return world * ne * args.steps * iw * ih / 1e6 / float(tt.item()), h_out

        v_pinned, h_out = e2e_leg(True)
        h2d = ne * iw * ih * 4 + (ne * ow * oh * 4 if wl["compose"] == 1 else 0)
        e2e = {"value": v_pinned, "unit": "Mpx/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": ne * ow * oh * 4, "images_per_step": ne,
               "host_memory": "pinned", "bound": "host link (PCIe): the kernel is not what limits this number",
               "h2d_gb_per_s": v_pinned * 4 / 1e3 / world,
               "api": "ifb200_scale_and_render_many (host buffers; uploads/kernels/downloads pipelined on 3 streams; returns when all results are in host memory)"}
        if rank == 0 and check is not None and w.canvas0 is None:
            check["e2e_vs_device_max_abs_delta"] = int(np.abs(h_out[0].numpy().astype(np.int16) - w.out[0].cpu().numpy().astype(np.int16)).max())
        v_pageable, _ = e2e_leg(False)
        e2e["pageable"] = {"value": v_pageable, "unit": "Mpx/s", "host_memory": "pageable (what Bitmap buffers are: aligned_buffer.rs:40-43)"}

    # ---- the other configurations of BASELINE.json at their own batch sizes on the same GPU (rank 0 of a 1-GPU run): driver-visible numbers
    others = None
    if rank == 0 and world == 1 and not args.no_others and args.workload == DEFAULT_WORKLOAD:
        others = {}
        w.close()
        for name, nb in (("c2_4k_to_512_lanczos3", 0), ("c3_8k_to_1080p_robidoux_sharpen", 0), ("c4_1080p_to_4k_mitchell_sepia_over", 0)):   # 0: the configuration's own batch
            try:
                ow_ = DeviceWorkload(args, name, local, batch_override=nb)
                ow_.warm(3, seconds=0.3)
                torch.cuda.synchronize()
                _e0, _e1, kev, hms = ow_.timed(max(3, args.steps // 2))
                torch.cuda.synchronize()
                rf = ow_.roofline([a.elapsed_time(b) for a, b in kev], hms)
                ck = ow_.check(args.content, 1) if not args.no_check else None
                others[name] = {"images_per_step": ow_.B, "input_mpx_per_s": ow_.B * ow_.wl["in_wh"][0] * ow_.wl["in_wh"][1] / 1e6 / (rf["kernel_ms"] / 1e3),
                                "roofline": {k: rf[k] for k in ("bound", "achieved", "peak", "unit", "frac", "kernel_ms", "kernel_ms_min", "algorithmic_bytes_per_launch",
                                                                "fused_jobs", "generic_jobs", "tile_jobs")},
                                "parity_check": ck}
                ow_.close()
            except Exception as e:                      # a failure here must not take the headline down with it
                others[name] = {"error": str(e)[:300]}

    if rank == 0:
        line = {"metric": "input Mpixels/s, " + args.workload, "value": value, "unit": "Mpx/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": total_ms_max / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_dict(args, wl, alpha, B),
                "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
                "parity_check": check, "out_mpx_per_s": world * B * args.steps * ow * oh / 1e6 / (total_ms_max / 1e3),
                "other_workloads": others, "git": git_sha()}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
