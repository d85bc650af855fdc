#!/usr/bin/env python
"""bench.py — benchmark of the hot path (driver contract: ONE JSON line on stdout).

Headline workload (BASELINE.json configs[1]): torchvision.ops.roi_align, 256-ch 200x272 fp32 FPN feature map, 1000 RoIs,
7x7 output, spatial_scale 0.25, sampling_ratio 2.  A "step" = one roi_align call over one such batch through the
reference-facing API (torchvision.ops.roi_align after vision_b200.install() -> dispatcher -> C ABI -> sm_100a kernels).
The other BASELINE configurations are measured in the same run as first-class blocks under "configs" (each with its own
`value`, `roofline`, `cpu_baseline`, `e2e`, and `gpu_reference` = the reference's own sm_100 CUDA kernels from the installed
wheel, same inputs, same box):
    cfg3  batched_nms   100k boxes x 80 classes per image, fp32, 4 images per rank          boxes/s
    cfg4  deform_conv2d 3x3, N=32 C=512->512 64x64, bf16 (tcgen05 path)                      TFLOP/s
    cfg5  resize        bilinear antialias, 128 x 3x2160x3840 fp16 -> 224x224 per rank       images/s

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--configs 2,3,4,5] [--dump-outputs DIR]
  torchrun --nproc-per-node N ... bench.py --gpus N ...      (one rank per GPU, NCCL)

N > 1 is weak scaling: every rank owns its own images.  Images are independent units, so the timed step has NO
data-path collective (tier rule 5); the north-star's exchange - an all-gather of the per-shard outputs - is measured next
to it as "with_allgather": the op is cut into chunks and each chunk's all-gather runs on a side stream under the next
chunk's kernel (vision_b200/sharded.py).  Each rank pins itself to the CPUs of its GPU's NUMA node before it allocates
pinned host memory (the e2e leg moves ~100 MB per step per rank through the host).

Timing: W >= 3 warm-up steps; L2 is flushed (256 MiB write) before every timed step; each step is bracketed by CUDA
events on the launching stream and the K step times are summed; barrier + synchronize on both sides; max over ranks.
Every timed loop of this project's path (headline, configs, e2e, all-gather legs) runs K steps; the legs that time the
reference keep their own small sample sizes.
`--dump-outputs DIR` writes, on rank 0, what the last timed step of each measured op returned as DIR/<name>.npy: the
headline roi_align output in full, and of the configs' larger outputs a fixed sample of DUMP_SAMPLE elements at seeded
positions (float32; integer results as float64).  The inputs are seeded, so two builds run with the same arguments can
be compared output for output.
`--impl reference` times the reference's own CPU kernel of the headline op (installed torchvision wheel; the oracle port
if it is absent) on the host cores.
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ALG_BYTES = 55_705_600 + 20_000 + 50_176_000      # map + rois + output (SURVEY.md §8d cfg2)
K_ROIS = 1000
# dram__bytes_read.sum + dram__bytes_write.sum of the headline kernel, one launch of this workload (profiles/, ncu --set full)
NCU_TRAFFIC = {"bytes": 67_071_744 + 9_524_224, "source": "profiles/r2_roi_align.ncu-rep / r2_roi_align_ncu.txt (ncu --set full, one launch; most of "
                                                          "the 50 MB output is still dirty in L2 when the capture ends)"}
# per-launch DRAM traffic of the dominant kernel of the other configs, same kind of capture (profiles/r2_*_ncu.txt)
NCU_TRAFFIC_CFG = {
    "cfg3": {"bytes": 1_622_784 + 8_721_664, "source": "profiles/r2_bnms_mask_ncu.txt + r2_bnms_scan_ncu.txt (one image)"},
    "cfg4": {"bytes": 146_062_848 + 97_087_488, "source": "profiles/r2_deform_bf16.ncu-rep / r2_deform_bf16_ncu.txt (deform_conv2d_tc_kernel, N=32)"},
    "cfg5": {"bytes": 6_426_276_000 + 42_117_888, "source": "profiles/r2_resize128.ncu-rep / r2_resize128_ncu.txt (resize_aa_stream_kernel, 128 images)"},
}
WORKLOAD = "roi_align fp32 1x256x200x272, 1000 RoIs, 7x7, scale 0.25, sampling_ratio 2, aligned=False (BASELINE configs[1])"
CFG3_IMAGES = 4
CFG3_BOXES = 100_000
CFG4_FLOPS = 2 * 32 * 64 * 64 * 512 * 512 * 9          # SURVEY.md §8d cfg4: 618,475,290,624
CFG5_BATCH = 128
CFG5_BYTES_PER_IMAGE = 3 * 2160 * 3840 * 2 + 3 * 224 * 224 * 2
DUMP_SAMPLE = 1 << 20            # elements kept of a config output larger than this (--dump-outputs)
DUMP_LIMIT = 64 << 20            # bytes written by --dump-outputs in all: 50.2 MB headline + <= 3.2 MB cfg3 + 2 x 4.2 MB samples


def _peaks_json() -> dict:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            pass
    return {}


def peaks():
    d = _peaks_json()
    if "hbm_gbs" in d:
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def tensor_peaks():
    d = _peaks_json()
    if "bf16_tflops" in d:
        return float(d["bf16_tflops"]), float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "measured (MEASURED_PEAKS.json)"
    return 1680.0, 1460.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def pin_to_gpu_numa(torch, local_rank: int) -> dict:
    """Bind this process to the CPUs local to its GPU (sysfs local_cpulist of the PCI device) BEFORE pinned buffers are
    allocated, so first-touch puts them on the GPU's NUMA node."""
    info = {"numa_node": None, "cpus": None}
    try:
        p = torch.cuda.get_device_properties(local_rank)
        base = f"/sys/bus/pci/devices/{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(base + "/numa_node").read().strip())
        cpulist = open(base + "/local_cpulist").read().strip()
        cpus = set()
        for part in cpulist.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        allowed = os.sched_getaffinity(0)
        cpus = (cpus & allowed) or allowed
        os.sched_setaffinity(0, cpus)
        info = {"numa_node": node, "cpus": len(cpus)}
    except Exception as ex:   # not fatal: containers may hide sysfs
        info["error"] = repr(ex)[:120]
    return info


# ------------------------------------------------------------------------------------------------------------------
# reference arm (CPU) of the headline op
# ------------------------------------------------------------------------------------------------------------------
def cpu_reference_fn():
    """The reference's own CPU implementation of the path, if the wheel is importable; else the oracle port.
    Returns (fn, kind, description, threads).  The reference kernel is a single-threaded loop over RoIs
    (csrc/ops/cpu/roi_align_kernel.cpp:33-35), so "all the host threads it can use" is one thread per call; to
    give it the whole machine the RoIs are split into one chunk per core and the UNMODIFIED op is called on the
    chunks from a thread pool (the op releases the GIL; outputs are concatenated in RoI order)."""
    import torch
    from concurrent.futures import ThreadPoolExecutor
    from vision_b200 import workloads

    x, rois, kw = workloads.cfg2_roi_align()
    threads = max(1, min(len(os.sched_getaffinity(0)), os.cpu_count() or 1, 64, rois.shape[0]))
    chunks = [c for c in torch.chunk(rois, threads, dim=0) if c.shape[0]]
    pool = ThreadPoolExecutor(max_workers=len(chunks))
    try:
        import torchvision

        def fn():
            return torch.cat(list(pool.map(lambda r: torchvision.ops.roi_align(x, r, **kw), chunks)), dim=0)

        return fn, "reference", (f"torchvision {torchvision.__version__} CPU kernel (csrc/ops/cpu/roi_align_kernel.cpp, a "
                                 f"single-threaded loop) called on {len(chunks)} RoI chunks from {len(chunks)} threads"), len(chunks)
    except Exception:
        import numpy as np
        import oracle

        xn = x.numpy()
        rn = [c.numpy() for c in chunks]

        def fn():
            return np.concatenate(list(pool.map(lambda r: oracle.roi_align(xn, r, kw["output_size"], kw["spatial_scale"],
                                                                         kw["sampling_ratio"], kw["aligned"]), rn)), axis=0)

        return fn, "port", f"oracle/vision_oracle.c restatement (single-threaded C) on {len(chunks)} RoI chunks / threads", len(chunks)


def time_cpu(fn, calls: int) -> float:
    fn()
    t0 = time.perf_counter()
    for _ in range(calls):
        fn()
    return (time.perf_counter() - t0) / calls


def run_reference(args, rank: int):
    if rank != 0:
        return
    import torch

    torch.set_num_threads(1)          # the pool supplies the parallelism; no intra-op threads under it
    fn, kind, desc, threads = cpu_reference_fn()
    for _ in range(min(args.warmup, 2)):
        fn()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = fn()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        write_outputs(args.dump_outputs, {"cfg2_roi_align": host_array(torch.as_tensor(out))})
    ms = dt / args.steps * 1e3
    val = K_ROIS / (ms / 1e3)
    line = {
        "impl": "reference", "metric": "roi_align RoIs/s", "value": val, "unit": "RoIs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "l2": "n/a (CPU)", "parallelism": "host cores"},
        "cpu_baseline": {"value": val, "unit": "RoIs/s", "cores": threads, "host_cores": os.cpu_count(), "kind": kind,
                         "sample": f"{args.steps} full-size calls of the workload; {desc}"},
        "e2e": {"value": val, "unit": "RoIs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# measurement helpers (product arm)
# ------------------------------------------------------------------------------------------------------------------
def host_array(t, sample=None):
    """`t` on the host as float32 (integer results as float64, which holds them exactly).  With `sample`, an output of more
    elements keeps only `sample` of them, flattened, at positions drawn from a fixed seed: the same positions in every run."""
    import numpy as np
    import torch

    t = t.detach()
    if sample is not None and t.numel() > sample:
        pos = np.sort(np.random.default_rng(0).choice(t.numel(), sample, replace=False))
        t = t.reshape(-1)[torch.from_numpy(pos).to(t.device)]
    t = t.cpu()
    return (t.float() if t.is_floating_point() else t.double()).numpy()


def write_outputs(path: str, arrays: dict) -> None:
    import numpy as np

    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


class Ctx:
    def __init__(self, torch, dist, dev, rank, world, args):
        self.torch, self.dist, self.dev, self.rank, self.world, self.args = torch, dist, dev, rank, world, args
        self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
        self.last = None                                      # what the last timed step of device_ms returned
        self.outputs = {} if args.dump_outputs and rank == 0 else None

    def keep_output(self, name: str, t, sample=None):
        """Keeps a host copy of `t` for --dump-outputs (rank 0 only)."""
        if self.outputs is not None:
            self.outputs[name] = host_array(t, sample)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v: float) -> float:
        if self.world == 1:
            return float(v)
        t = self.torch.tensor([v], device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def device_ms(self, fn, steps: int, warmup: int = 3, flush: bool = True) -> float:
        """ms per step: L2 flushed before every step, per-step CUDA events on the current stream, summed; max over ranks."""
        torch = self.torch
        for _ in range(warmup):
            if flush:
                self.flush.zero_()
            fn()
        self.barrier()
        stream = torch.cuda.current_stream()
        starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        for i in range(steps):
            if flush:
                self.flush.zero_()
            self.last = None                  # the previous step's output is freed before this step, as when nothing keeps it
            starts[i].record(stream)
            self.last = fn()
            ends[i].record(stream)
        self.barrier()
        return self.max_over_ranks(sum(s.elapsed_time(e) for s, e in zip(starts, ends)) / steps)

    def e2e_ms(self, host_inputs, op, out_numel_dtype, steps: int):
        """End to end through the public API: EVERY step copies its inputs from pinned host memory to the device and its
        result back.  Three streams (copy-in / compute / copy-out) with double buffers, so step i's D2H overlaps step i+1's
        H2D (PCIe is full duplex); all copies stay inside the timed region.  Returns (ms per step, h2d bytes, d2h bytes)."""
        torch = self.torch
        dev = self.dev
        hin = [t.pin_memory() if not t.is_pinned() else t for t in host_inputs]
        dbuf = [[torch.empty(t.shape, dtype=t.dtype, device=dev) for t in hin] for _ in range(2)]
        numel, odt = out_numel_dtype
        hout = [torch.empty(numel, dtype=odt).pin_memory() for _ in range(2)]
        s_in, s_cmp, s_out = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
        ev_in = [torch.cuda.Event() for _ in range(2)]
        ev_cmp = [torch.cuda.Event() for _ in range(2)]
        ev_out = [torch.cuda.Event() for _ in range(2)]
        d2h = [0]

        def run(n):
            for i in range(n):
                b = i % 2
                with torch.cuda.stream(s_in):
                    if i >= 2:
                        s_in.wait_event(ev_cmp[b])            # device input buffers free again
                    for d, h in zip(dbuf[b], hin):
                        d.copy_(h, non_blocking=True)
                    ev_in[b].record(s_in)
                with torch.cuda.stream(s_cmp):
                    s_cmp.wait_event(ev_in[b])
                    o = op(*dbuf[b])
                    ev_cmp[b].record(s_cmp)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev_cmp[b])
                    o.record_stream(s_out)
                    flat = o.reshape(-1)
                    hout[b][:flat.numel()].copy_(flat, non_blocking=True)
                    d2h[0] = flat.numel() * flat.element_size()
                    ev_out[b].record(s_out)

        torch.cuda.synchronize()
        run(4)
        self.barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(s_in)
        run(steps)
        e.record(s_out)
        torch.cuda.synchronize()
        ms = self.max_over_ranks(s.elapsed_time(e) / steps)
        h2d = sum(t.numel() * t.element_size() for t in hin)
        return ms, h2d, d2h[0]


def gpu_reference_ms(ctx: Ctx, vb, fn, steps: int, warmup: int = 2) -> float:
    """`fn` through the reference's own CUDA kernels: our CUDA-key override is removed for the duration."""
    was = vb.installed()
    if was:
        vb.uninstall()
    try:
        return ctx.device_ms(fn, steps, warmup)
    finally:
        if was:
            vb.install()


def block_cfg3(ctx: Ctx, vb, tv, sharded) -> dict:
    torch = ctx.torch
    from vision_b200 import workloads

    imgs = [workloads.cfg3_batched_nms(seed=ctx.rank * CFG3_IMAGES + j) for j in range(CFG3_IMAGES)]
    dimgs = [tuple(t.to(ctx.dev) for t in im) for im in imgs]
    steps = ctx.args.steps
    kept = [0]

    def step():
        keep = [tv.ops.batched_nms(b, s, i, 0.5) for (b, s, i) in dimgs]
        kept[0] = sum(int(k.numel()) for k in keep)
        return keep

    ms = ctx.device_ms(step, steps)
    for j, k in enumerate(ctx.last):
        ctx.keep_output(f"cfg3_batched_nms_keep_image{j}", k)
    boxes = ctx.world * CFG3_IMAGES * CFG3_BOXES
    alg = CFG3_IMAGES * (CFG3_BOXES * (16 + 4 + 8)) + 8 * kept[0]
    peak, src = peaks()
    cl = workloads.cfg3_batched_nms(seed=1000 + ctx.rank, clustered=True)
    cld = tuple(t.to(ctx.dev) for t in cl)
    ms_cl = ctx.device_ms(lambda: tv.ops.batched_nms(*cld, 0.5), steps)
    out = {
        "metric": "batched_nms boxes/s", "value": boxes / (ms / 1e3), "unit": "boxes/s", "ms_per_step": ms, "steps": steps, "dtype": "f32",
        "config": {"workload": f"batched_nms fp32, {CFG3_BOXES} boxes x 80 classes per image (uniform boxes, distinct scores), "
                               f"{CFG3_IMAGES} images per rank, iou 0.5 (BASELINE configs[2]); reference strategy: per-class (numel > 100k)",
                   "api": "torchvision.ops.batched_nms after vision_b200.install() (one host sync per image for the output size)",
                   "l2": "flushed before every timed step"},
        "ms_per_image": ms / CFG3_IMAGES, "clustered_ms_per_image": ms_cl,
        "roofline": {"bound": "hbm", "achieved": alg / (ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": alg / (ms / 1e3) / 1e9 / peak, "traffic": NCU_TRAFFIC_CFG["cfg3"]["bytes"] * CFG3_IMAGES,
                     "traffic_source": NCU_TRAFFIC_CFG["cfg3"]["source"], "algorithmic_bytes": alg, "peak_source": src,
                     "note": "HBM-nominal only: 2.8 MB per image is < 1 us of HBM time; the real bound is the per-class greedy chain plus "
                             "sum n_c^2/2 = 62.5 M IoU tests per image (DESIGN.md 4.3)",
                     "iou_pairs_per_s": ctx.world * CFG3_IMAGES * 62.5e6 / (ms / 1e3)},
    }
    # e2e: one image per step
    b, s, i = imgs[0]
    ems, h2d, d2h = ctx.e2e_ms([b, s, i], lambda bb, ss, ii: tv.ops.batched_nms(bb, ss, ii, 0.5), (CFG3_BOXES, torch.int64), steps)
    out["e2e"] = {"value": ctx.world * CFG3_BOXES / (ems / 1e3), "unit": "boxes/s", "ms_per_step": ems, "h2d_bytes_per_step": h2d,
                  "d2h_bytes_per_step": d2h, "note": "one image per step: pinned host -> H2D -> batched_nms -> D2H of the kept indices"}
    if ctx.world > 1:
        gms = ctx.device_ms(lambda: sharded.sharded_batched_nms_padded(dimgs, 0.5), steps)
        out["with_allgather"] = {"ms_per_step": gms, "value": boxes / (gms / 1e3), "unit": "boxes/s",
                                 "bytes_gathered_per_rank": ctx.world * CFG3_IMAGES * (CFG3_BOXES + 1) * 8,
                                 "note": "sharded_batched_nms_padded: no host sync, ONE all_gather_into_tensor of the padded keep lists"}
    if ctx.rank == 0 and ctx.world == 1:
        g = gpu_reference_ms(ctx, vb, lambda: tv.ops.batched_nms(*dimgs[0], 0.5), 3, 1)
        out["gpu_reference"] = {"ms_per_image": g, "value": CFG3_BOXES / (g / 1e3), "unit": "boxes/s",
                                "ours_over_reference": g / (ms / CFG3_IMAGES),
                                "what": "torchvision.ops.batched_nms on the wheel's sm_100 kernels (per-class Python loop + nms_kernel_impl), same boxes"}
        from concurrent.futures import ThreadPoolExecutor
        torch.set_num_threads(1)
        nthr = min(len(os.sched_getaffinity(0)), 16)
        cpu_imgs = [workloads.cfg3_batched_nms(seed=50 + j) for j in range(nthr)]
        pool = ThreadPoolExecutor(max_workers=nthr)
        fn = lambda: list(pool.map(lambda im: tv.ops.batched_nms(im[0], im[1], im[2], 0.5), cpu_imgs))
        sec = time_cpu(fn, 2)
        out["cpu_baseline"] = {"value": nthr * CFG3_BOXES / sec, "unit": "boxes/s", "cores": nthr, "kind": "reference",
                               "sample": f"2 passes over {nthr} images ({sec:.2f} s each), the unmodified CPU op (single-threaded per call) on one image per thread"}
    return out


def block_cfg4(ctx: Ctx, vb, tv, sharded) -> dict:
    torch = ctx.torch
    from vision_b200 import workloads

    x, off, w, b, m = workloads.cfg4_deform_conv2d(device=ctx.dev, seed=ctx.rank)
    steps = ctx.args.steps
    op = lambda: tv.ops.deform_conv2d(x, off, w, b, 1, 1, 1, m)
    ms = ctx.device_ms(op, steps)
    ctx.keep_output("cfg4_deform_conv2d_sample", ctx.last, DUMP_SAMPLE)
    tf = CFG4_FLOPS / (ms / 1e3) / 1e12
    burst, sustained, src = tensor_peaks()
    out = {
        "metric": "deform_conv2d TFLOP/s", "value": ctx.world * tf, "unit": "TFLOP/s", "ms_per_step": ms, "steps": steps, "dtype": "bf16",
        "config": {"workload": "deform_conv2d 3x3 DCNv2, N=32 C=512->512 64x64, stride 1 pad 1, bf16 in / fp32 accumulate (BASELINE configs[3])",
                   "api": "torchvision.ops.deform_conv2d after vision_b200.install()", "l2": "flushed before every timed step",
                   "includes": "NCHW->NHWC staging of the input and weight packing (re-done every call) + the tcgen05 kernel"},
        "roofline": {"bound": "tensor", "achieved": tf, "peak": burst, "unit": "TFLOP/s", "frac": tf / burst,
                     "frac_of_sustained": tf / sustained, "peak_sustained": sustained, "traffic": NCU_TRAFFIC_CFG["cfg4"]["bytes"],
                     "traffic_source": NCU_TRAFFIC_CFG["cfg4"]["source"], "tensor_pipe_active_pct_ncu": 52.7,
                     "algorithmic_flops": CFG4_FLOPS, "peak_source": src + " (burst: the op is timed alone between L2 flushes)"},
    }
    hx, hoff, hw_, hb, hm = [t.cpu() for t in (x, off, w, b, m)]
    ems, h2d, d2h = ctx.e2e_ms([hx, hoff, hw_, hb, hm], lambda a, o, ww, bb, mm: tv.ops.deform_conv2d(a, o, ww, bb, 1, 1, 1, mm),
                               (x.numel(), torch.bfloat16), steps)
    out["e2e"] = {"value": ctx.world * CFG4_FLOPS / (ems / 1e3) / 1e12, "unit": "TFLOP/s", "ms_per_step": ems, "h2d_bytes_per_step": h2d,
                  "d2h_bytes_per_step": d2h}
    if ctx.world > 1:
        g = sharded.OverlappedGather()
        part = lambda i: tv.ops.deform_conv2d(x[i * 8:(i + 1) * 8], off[i * 8:(i + 1) * 8], w, b, 1, 1, 1, m[i * 8:(i + 1) * 8])
        gms = ctx.device_ms(lambda: g.run(part, 4), steps)
        nccl = {"ms_per_step": gms, "value": ctx.world * CFG4_FLOPS / (gms / 1e3) / 1e12, "unit": "TFLOP/s",
                "bytes_gathered_per_rank": ctx.world * x.numel() * 2,
                "note": "4 batch chunks, each chunk's all_gather_into_tensor on a side stream under the next chunk's kernel"}
        out["with_allgather"] = nccl
        peer = sharded.PeerGather.create(tuple(x.shape), x.dtype, ctx.dev)      # C_out = C_in, same spatial size: output shard = input shape
        if ctx.max_over_ranks(0.0 if peer is not None else 1.0) == 0.0:
            want = sharded.all_gather_equal(op())
            got = sharded.deform_conv2d_gather(x, off, w, b, peer, 1, 1, 1, m)
            same = bool(torch.equal(got, want))
            fms = ctx.device_ms(lambda: sharded.deform_conv2d_gather(x, off, w, b, peer, 1, 1, 1, m), steps)
            ingress = (ctx.world - 1) * x.numel() * 2
            if same:                          # a fused result that differs from the NCCL gather would be reported, never adopted
                out["with_allgather"] = {
                    "ms_per_step": fms, "value": ctx.world * CFG4_FLOPS / (fms / 1e3) / 1e12, "unit": "TFLOP/s",
                    "bytes_gathered_per_rank": ctx.world * x.numel() * 2, "identical_to_nccl_gather": True,
                    "nvlink_ingress_floor_ms": ingress / 900e9 * 1e3,
                    "note": "all-gather fused into the tcgen05 kernel's epilogue: each output element is stored to every rank's gathered buffer "
                            "(torch symmetric memory, NVLink peer stores of 256-byte runs), one device-side barrier per step (double-buffered); "
                            "no NCCL call.  nvlink_ingress_floor_ms = (world-1) x 134 MB received per rank per step at 900 GB/s",
                    "nccl_overlapped": nccl}
            else:
                nccl["fused_peer_stores"] = {"ms_per_step": fms, "identical_to_nccl_gather": False}
            del want, got
        else:
            out["with_allgather"]["peer_stores"] = "unavailable on this box (symmetric memory rendezvous failed); NCCL exchange reported"
        del peer
    if ctx.rank == 0 and ctx.world == 1:
        xf, of, wf, bf, mf = x.float(), off.float(), w.float(), b.float(), m.float()
        old = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = False
        try:
            g32 = gpu_reference_ms(ctx, vb, lambda: tv.ops.deform_conv2d(xf, of, wf, bf, 1, 1, 1, mf), 3, 1)
        finally:
            torch.backends.cuda.matmul.allow_tf32 = old
        del xf, of, wf, bf, mf
        xh, oh, wh, bh, mh = x.half(), off.half(), w.half(), b.half(), m.half()
        g16 = gpu_reference_ms(ctx, vb, lambda: tv.ops.deform_conv2d(xh, oh, wh, bh, 1, 1, 1, mh), 5, 1)
        del xh, oh, wh, bh, mh
        out["gpu_reference"] = {"fp32_ms": g32, "fp16_ms": g16, "value": CFG4_FLOPS / (g16 / 1e3) / 1e12, "unit": "TFLOP/s",
                                "ours_over_reference": g16 / ms, "ours_over_reference_fp32": g32 / ms,
                                "what": "torchvision.ops.deform_conv2d on the wheel's sm_100 kernels (im2col + cuBLAS), same values; the reference "
                                        "has no bf16 kernel, so its fastest 16-bit option (fp16, inputs pre-cast) and its fp32 default are both timed"}
        torch.set_num_threads(len(os.sched_getaffinity(0)))
        cx, coff, cw, cb, cm = [t[:2].float().cpu() if t.dim() == 4 and t.shape[0] == 32 else t.float().cpu() for t in (x, off, w, b, m)]
        sec = time_cpu(lambda: tv.ops.deform_conv2d(cx, coff, cw, cb, 1, 1, 1, cm), 1)
        out["cpu_baseline"] = {"value": CFG4_FLOPS / 16 / sec / 1e12, "unit": "TFLOP/s", "cores": torch.get_num_threads(), "kind": "reference",
                               "sample": f"N=2 of the 32 images (1/16 of the workload), fp32, {sec:.2f} s per call: single-threaded im2col + MKL GEMM"}
    return out


def block_cfg5(ctx: Ctx, vb, tv, sharded) -> dict:
    torch = ctx.torch
    from torchvision.transforms.v2 import functional as TF
    from vision_b200 import workloads

    x = workloads.cfg5_resize(device=ctx.dev, batch=CFG5_BATCH, seed=ctx.rank)
    steps = ctx.args.steps
    ms = ctx.device_ms(lambda: TF.resize(x, [224, 224]), steps)
    ctx.keep_output("cfg5_resize_sample", ctx.last, DUMP_SAMPLE)
    nbytes = CFG5_BATCH * CFG5_BYTES_PER_IMAGE
    peak, src = peaks()
    out = {
        "metric": "resize images/s", "value": ctx.world * CFG5_BATCH / (ms / 1e3), "unit": "images/s", "ms_per_step": ms, "steps": steps,
        "dtype": "f16 storage, f32 arithmetic",
        "config": {"workload": f"resize bilinear antialias, {CFG5_BATCH} x 3x2160x3840 fp16 -> 224x224 per rank (the per-GPU shard of BASELINE "
                               f"configs[4] at 8 GPUs; 1024 images = 8 such shards)",
                   "api": "torchvision.transforms.v2.functional.resize after vision_b200.install()", "l2": "input (6.4 GB) exceeds L2; flushed anyway"},
        "roofline": {"bound": "hbm", "achieved": nbytes / (ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": nbytes / (ms / 1e3) / 1e9 / peak, "traffic": NCU_TRAFFIC_CFG["cfg5"]["bytes"],
                     "traffic_source": NCU_TRAFFIC_CFG["cfg5"]["source"], "algorithmic_bytes": nbytes, "peak_source": src},
    }
    sub = 32
    hx = x[:sub].cpu()
    ems, h2d, d2h = ctx.e2e_ms([hx], lambda a: TF.resize(a, [224, 224]), (sub * 3 * 224 * 224, torch.float16), steps)
    out["e2e"] = {"value": ctx.world * sub / (ems / 1e3), "unit": "images/s", "ms_per_step": ems, "h2d_bytes_per_step": h2d,
                  "d2h_bytes_per_step": d2h, "note": f"{sub} images per step (1.6 GB of pinned host memory), H2D-bound"}
    del hx
    if ctx.world > 1:
        g = sharded.OverlappedGather()
        gms = ctx.device_ms(lambda: sharded.sharded_apply_overlapped(lambda t: TF.resize(t, [224, 224]), x, chunks=4, gather=g), steps)
        nccl = {"ms_per_step": gms, "value": ctx.world * CFG5_BATCH / (gms / 1e3), "unit": "images/s",
                "bytes_gathered_per_rank": ctx.world * CFG5_BATCH * 3 * 224 * 224 * 2,
                "note": "4 chunks of 32 images, each chunk's all_gather_into_tensor on a side stream under the next chunk's kernel"}
        out["with_allgather"] = nccl
        # the exchange fused into the kernel: every output pixel is stored to all ranks' gathered buffers (peer-mapped memory)
        peer = sharded.PeerGather.create((CFG5_BATCH, 3, 224, 224), x.dtype, ctx.dev)
        ok = ctx.max_over_ranks(0.0 if peer is not None else 1.0) == 0.0      # every rank must have it
        if ok:
            want = sharded.sharded_apply_overlapped(lambda t: TF.resize(t, [224, 224]), x, chunks=4, gather=g).materialize()
            got = sharded.resize_gather(x, [224, 224], peer)
            same = bool(torch.equal(got, want))
            fms = ctx.device_ms(lambda: sharded.resize_gather(x, [224, 224], peer), steps)
            if same:
                out["with_allgather"] = {
                    "ms_per_step": fms, "value": ctx.world * CFG5_BATCH / (fms / 1e3), "unit": "images/s",
                    "bytes_gathered_per_rank": ctx.world * CFG5_BATCH * 3 * 224 * 224 * 2, "identical_to_nccl_gather": True,
                    "note": "all-gather fused into the resize kernel: each finished pixel is stored to every rank's gathered buffer (torch symmetric "
                            "memory, NVLink peer stores), one device-side barrier per step (double-buffered); no NCCL call",
                    "nccl_overlapped": nccl}
            else:
                nccl["fused_peer_stores"] = {"ms_per_step": fms, "identical_to_nccl_gather": False}
            del want, got
        else:
            out["with_allgather"]["peer_stores"] = "unavailable on this box (symmetric memory rendezvous failed); NCCL exchange reported"
        del peer
    if ctx.rank == 0 and ctx.world == 1:
        xs = x[:sub]
        g = gpu_reference_ms(ctx, vb, lambda: TF.resize(xs, [224, 224]), 3, 1)
        out["gpu_reference"] = {"ms_per_32_images": g, "value": sub / (g / 1e3), "unit": "images/s",
                                "ours_over_reference": (g / sub) / (ms / CFG5_BATCH),
                                "what": "the reference route on this GPU: fp16 -> fp32 cast, aten::_upsample_bilinear2d_aa, cast back (32 images per call: "
                                        "its fp32 temporary is 2x the input)"}
        rows = {}
        for name, kw in (("bicubic_antialias", dict(interpolation=TF.InterpolationMode.BICUBIC)), ("bilinear_no_antialias", dict(antialias=False))):
            o = ctx.device_ms(lambda: TF.resize(xs, [224, 224], **kw), steps)
            r = gpu_reference_ms(ctx, vb, lambda: TF.resize(xs, [224, 224], **kw), 2, 1)
            rows[name] = {"ms_per_32_images": o, "reference_ms_per_32_images": r, "ours_over_reference": r / o}
        out["secondary_modes"] = rows
        torch.set_num_threads(len(os.sched_getaffinity(0)))
        cx = x[:8].cpu()
        sec = time_cpu(lambda: TF.resize(cx, [224, 224]), 1)
        out["cpu_baseline"] = {"value": 8 / sec, "unit": "images/s", "cores": torch.get_num_threads(), "kind": "reference",
                               "sample": f"8 images ({sec:.2f} s per call): the unmodified v2 resize on CPU tensors (cast + ATen upsample_bilinear2d_aa, all cores)"}
    del x
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50, help="timed steps of every measurement of this project's path")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-secondary", action="store_true", help="headline (cfg2) only")
    ap.add_argument("--configs", default="2,3,4,5", help="which BASELINE configs to measure (2 is always measured)")
    ap.add_argument("--cpu-calls", type=int, default=10, help="CPU-baseline sample size (full-size calls)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step of each measured op returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist

    assert args.warmup >= 3, "timing rules: W >= 3"
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback on the product path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # single rank: nothing competes for the host, and the CPU baseline should see every core
    numa = pin_to_gpu_numa(torch, local_rank) if world > 1 else {"skipped": "single rank"}
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import torchvision
    import vision_b200 as vb
    from vision_b200 import sharded, workloads

    vb.install()
    ctx = Ctx(torch, dist, dev, rank, world, args)
    x, rois, kw = workloads.cfg2_roi_align(seed=rank)
    xd, rd = x.to(dev), rois.to(dev)
    flush = ctx.flush
    stream = torch.cuda.current_stream()

    def step():
        return torchvision.ops.roi_align(xd, rd, **kw)

    for _ in range(args.warmup):
        flush.zero_()
        step()
    ctx.barrier()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    launches0 = vb.launch_count()
    wall0 = time.perf_counter()
    for i in range(args.steps):
        flush.zero_()                       # L2 flush between timed iterations (not timed)
        out = None                          # the previous step's output is freed before this step, as when nothing keeps it
        starts[i].record(stream)
        out = step()
        ends[i].record(stream)
    ctx.barrier()
    wall = time.perf_counter() - wall0
    launches = vb.launch_count() - launches0
    ctx.keep_output("cfg2_roi_align", out)
    del out
    ms_per_step = ctx.max_over_ranks(sum(s.elapsed_time(e) for s, e in zip(starts, ends))) / args.steps

    # ---- end to end: pinned host buffers; EVERY step copies its inputs H2D and its result D2H ----
    e2e_ms, h2d, d2h = ctx.e2e_ms([x, rois], lambda a, r: torchvision.ops.roi_align(a, r, **kw), (K_ROIS * 256 * 49, torch.float32), args.steps)

    # ---- the all-gather of per-shard outputs (N > 1), hidden behind the kernel ----
    # The op is cut along CHANNELS (4 x 64 planes: each chunk's input slice is contiguous for one image, and a plane-resident
    # kernel does not re-stage planes as it would if the RoIs were cut); chunk i's all_gather_into_tensor runs on a side stream
    # under chunk i+1's kernel.  The gathered result is [chunks, world, K, 64, 7, 7]: rank r's channels [64 i, 64 i + 64) at [i, r].
    gather = None
    if world > 1:
        og = sharded.OverlappedGather()
        chunks = 4
        cper = xd.shape[1] // chunks
        xchunks = [xd[:, i * cper:(i + 1) * cper] for i in range(chunks)]
        assert all(c.is_contiguous() for c in xchunks)
        g_steps = args.steps
        gms = ctx.device_ms(lambda: og.run(lambda i: torchvision.ops.roi_align(xchunks[i], rd, **kw), chunks), g_steps)
        plain = ctx.device_ms(lambda: sharded.all_gather_equal(torchvision.ops.roi_align(xd, rd, **kw)), g_steps)
        best = min(gms, plain)
        gather = {"ms_per_step": best, "value": world * K_ROIS / (best / 1e3), "unit": "RoIs/s", "bytes_gathered_per_rank": world * K_ROIS * 256 * 49 * 4,
                  "overlapped_ms_per_step": gms, "serial_ms_per_step": plain,
                  "note": "op + all-gather of the per-shard outputs (NCCL).  overlapped = 4 channel chunks, chunk i's all_gather_into_tensor on a "
                          "side stream under chunk i+1's kernel; serial = one un-overlapped collective after the full op; ms_per_step = the better "
                          "of the two; L2 flushed before every step"}

        # the exchange fused into the kernel (vision_b200.sharded.PeerGather): every finished bin goes to all ranks' buffers, by one
        # NVSwitch multicast store where the box offers it, else by one NVLink peer store per rank
        peer = sharded.PeerGather.create((K_ROIS, 256, 7, 7), torch.float32, dev)
        if ctx.max_over_ranks(0.0 if peer is not None else 1.0) == 0.0:
            ref = sharded.all_gather_equal(torchvision.ops.roi_align(xd, rd, **kw))
            fused = {}
            for name, mc in (("multicast", True), ("peer_stores", False)):
                if mc and ctx.max_over_ranks(0.0 if peer.mc_ptr else 1.0) != 0.0:
                    continue
                try:
                    got = sharded.roi_align_gather(xd, rd, peer, multicast=mc, **kw)
                    same = bool(torch.equal(got, ref))
                    fms = ctx.device_ms(lambda: sharded.roi_align_gather(xd, rd, peer, multicast=mc, **kw), g_steps)
                    fused[name] = {"ms_per_step": fms, "value": world * K_ROIS / (fms / 1e3), "identical_to_nccl_gather": same}
                except Exception as ex:      # noqa: BLE001 - an unsupported transport must not take the line down
                    fused[name] = {"error": repr(ex)[:200]}
            ok = {k_: v for k_, v in fused.items() if v.get("identical_to_nccl_gather")}
            ingress = (world - 1) * K_ROIS * 256 * 49 * 4
            gather["nvlink_ingress_floor_ms"] = ingress / 900e9 * 1e3
            gather["fused_variants"] = fused
            gather["transport"] = "nccl"
            if ok:
                bname = min(ok, key=lambda k_: ok[k_]["ms_per_step"])
                if ok[bname]["ms_per_step"] < gather["ms_per_step"]:
                    gather.update({"ms_per_step": ok[bname]["ms_per_step"], "value": ok[bname]["value"], "transport": bname})
            gather["note"] += (".  fused_variants: the exchange done by the roi_align kernel's own stores into every rank's gathered buffer (torch symmetric "
                               "memory; multicast = one multimem.st replicated by the NVSwitch, peer_stores = one NVLink store per rank; 28-byte runs, "
                               "so the links carry partial sectors), one device-side barrier per step; ms_per_step / value = the fastest "
                               "transport.  Every rank RECEIVES (world-1) x 50 MB per step: nvlink_ingress_floor_ms is that volume at 900 GB/s, the "
                               "bound of this exchange whatever the transport")
            del ref
        else:
            gather["peer_stores"] = "unavailable on this box (symmetric memory rendezvous failed); NCCL exchange reported"
        del peer

    configs = {}
    want = set(args.configs.split(",")) if not args.no_secondary else set()
    for key, fn in (("3", block_cfg3), ("4", block_cfg4), ("5", block_cfg5)):
        if key not in want:
            continue
        name = {"3": "cfg3_batched_nms", "4": "cfg4_deform_conv2d", "5": "cfg5_resize"}[key]
        try:
            configs[name] = fn(ctx, vb, torchvision, sharded)
        except Exception as ex:       # a failing secondary block never takes the headline down (every rank reaches the barrier below)
            configs[name] = {"error": repr(ex)[:400]}
        ctx.barrier()

    # sampled from the first headline step to the end of the last block (the headline region alone lasts ~10 ms)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        peak, peak_src = peaks()
        achieved = ALG_BYTES / (ms_per_step / 1e3) / 1e9     # per GPU (every rank runs the same kernel on its own image)
        cpu = gpu_ref = None
        if world == 1:
            g = gpu_reference_ms(ctx, vb, lambda: torchvision.ops.roi_align(xd, rd, **kw), 10)
            gpu_ref = {"ms_per_step": g, "value": K_ROIS / (g / 1e3), "unit": "RoIs/s", "ours_over_reference": g / ms_per_step,
                       "what": "torchvision.ops.roi_align on the wheel's sm_100 kernel (roi_align_forward_kernel_impl), same inputs, L2 flushed"}
            torch.set_num_threads(1)      # the pool supplies the parallelism
            fn, kind, desc, threads = cpu_reference_fn()
            sec = time_cpu(fn, args.cpu_calls)
            cpu = {"value": K_ROIS / sec, "unit": "RoIs/s", "cores": threads, "host_cores": os.cpu_count(), "kind": kind,
                   "sample": f"{args.cpu_calls} full-size calls ({sec * 1e3:.0f} ms each); {desc}"}
        # the shared-memory gather floor of the op (DESIGN.md 4.1): 12.5 M bins x 16 taps x 4 B through 148 SMs x 128 B/clk
        smem_floor_us = 12_544_000 * 16 * 4 / (148 * 128 * 1.965e9) * 1e6
        line = {
            "metric": "roi_align RoIs/s", "value": world * K_ROIS / (ms_per_step / 1e3), "unit": "RoIs/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "l2": "flushed before every timed step (256 MiB write); per-step CUDA events summed",
                       "parallelism": f"dp{world}: one image per rank, no data-path collective in the timed step",
                       "api": "torchvision.ops.roi_align after vision_b200.install()", "numa": numa},
            "roofline": {
                "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": NCU_TRAFFIC["bytes"],
                "traffic_source": NCU_TRAFFIC["source"],
                "kernel": "roi_align_line_kernel<7, 2> (+ roi_align_line_geometry_kernel inside the same event pair)",
                "algorithmic_bytes": ALG_BYTES, "peak_source": peak_src,
                "smem_gather_floor_us": smem_floor_us, "frac_of_smem_gather_floor": smem_floor_us / (ms_per_step * 1e3),
                "note": "the op is a shared-memory gather (200 M tap reads): its conflict-free floor is above the HBM time (DESIGN.md 4.1)"},
            "cpu_baseline": cpu, "gpu_reference": gpu_ref,
            "e2e": {"value": world * K_ROIS / (e2e_ms / 1e3), "unit": "RoIs/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "note": "pinned host buffers (NUMA-local to the GPU), H2D + op + D2H every step; 3 streams, double-buffered"},
            "gpu_launches": int(launches), "clocks": clocks, "wall_s_timed_region": wall,
        }
        if gather is not None:
            line["with_allgather"] = gather
        if configs:
            line["configs"] = configs
        if ctx.outputs is not None:
            write_outputs(args.dump_outputs, ctx.outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
