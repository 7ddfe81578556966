#!/usr/bin/env python
"""Benchmark of the batched caption-inference hot path (metric of BASELINE.json: captioned images/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload c2|c3|c4] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch per GPU: images -> backbone+FPN+heads -> MT encoder ->
T KV-cached beam-search steps -> token ids.  Workload (N=1 and per-GPU for N>1, weak scaling) = config C2 of
BASELINE.json: ResNet-50-FPN + Multi-Transformer, beam 8, batch 64, 3x512x512 synthetic images U(-1,1),
random-init weights, V=10000, T=64 decode steps, early stop OFF (fixed work).

  value  images/s, inputs already resident in HBM, ids left on the device (+ NCCL all-gather of ids for N>1),
         through the streaming call with `--lanes` batches in flight per GPU (default 3: the encoder of batch i+1 runs
         under the decode of batch i; every batch is submitted and collected inside the timed region),
         timed with CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks.
  one_shot  the same batches one at a time through Engine.generate (the latency of a batch; ids equal to the streamed ones).
  e2e    images/s through the public streaming call (Engine.generate_stream == fpnmt_stage_images +
         fpnmt_generate_staged, what Pipeline.evaluate uses) with PINNED HOST images and host results: every step's
         H2D copy of its batch and D2H read of ids/lengths are inside the timed region; the copy of batch i+1 is
         overlapped with the compute of batch i.  e2e.unpipelined_value is the same through the one-shot
         Engine.generate (copy, compute, read back strictly in sequence).
  roofline      heaviest kernel of the step (tcgen05 implicit GEMM), algorithmic FLOPs / CUDA-event time, measured
                live by the engine's per-op profiler right after the timed region.
  cpu_baseline  the oracle's faithful restatement of the reference (per image, uncached decode) on the host cores.

--dump-outputs DIR writes what the timed streaming call returned for its last batch (all ranks' token ids and caption
lengths after the all-gather) as DIR/ids.npy and DIR/lens.npy in float64, so that two builds can be compared output for
output: weights and images are seeded, so the same arguments give the same inputs on every run.

--impl reference times that restated reference alone (TensorFlow is not installable here, so the "reference arm"
is the oracle port; DESIGN.md records this).
"""
from __future__ import annotations

import argparse
import json
import os

# stdout carries exactly one JSON line.  NCCL logs through NCCL_DEBUG_FILE, except the NCCL_DEBUG=VERSION banner, which is a
# bare printf to stdout: that level is mapped to WARN and the version is written to stderr by run_own instead.
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
_NCCL_BANNER = os.environ.get("NCCL_DEBUG", "").upper() == "VERSION"
if _NCCL_BANNER:
    os.environ["NCCL_DEBUG"] = "WARN"
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "fpn-mt-image-captioning_b200"))

WORKLOADS = {
    "c2": dict(backbone="resnet50", batch=64, beam=8, vocab=10000, max_len=64,
               name="C2: ResNet-50-FPN + Multi-Transformer, beam=8, batch 64/GPU, 3x512x512, V=10000, T=64, early stop off"),
    "c3": dict(backbone="mobilenet224_1.0", batch=256, beam=8, vocab=10000, max_len=64,
               name="C3: MobileNetV2-FPN + Multi-Transformer, beam=8, batch 256/GPU, 3x512x512, V=10000, T=64, early stop off"),
    "c4": dict(backbone="densenet121", batch=64, beam=8, vocab=10000, max_len=64,
               name="C4: DenseNet-121-FPN + Multi-Transformer, beam=8, batch 64/GPU, 3x512x512, V=10000, T=64, early stop off"),
}
F_ENC = {"resnet50": 100.30e9, "mobilenet224_1.0": 61.54e9, "densenet121": 89.47e9}   # SURVEY.md §8a totals, FLOP/image
F_DEC = 28.1e9                                                                        # N=8, T=64, V=1e4, KV-cached


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=d["hbm_gbs"], tf=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tf=1590.0, tf_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """SM clock / power / throttle reasons sampled every 50 ms on a thread while the timed region runs (NVML in
    process; `nvidia-smi` polling as the fallback)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index: int):
        self.idx, self.samples, self.started, self.how = gpu_index, [], False, None
        self.stop_flag = threading.Event()

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if self.idx < len(ids) and ids[self.idx].isdigit():
                return int(ids[self.idx])
        return self.idx

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.how = "nvml"
        except Exception:
            self.nv, self.how = None, "nvidia-smi"
        self.t = threading.Thread(target=self._poll, daemon=True)
        self.t.start()
        self.started = True

    def _poll(self):
        if self.nv is not None:
            nv = self.nv
            while not self.stop_flag.is_set():
                try:
                    sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                    pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                    try:
                        rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                    except Exception:
                        rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                    self.samples.append((sm, self.sm_max, pw, rs))
                except Exception:
                    pass
                self.stop_flag.wait(0.05)
            return
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        cmd = ["nvidia-smi", "-i", str(self._physical_index()), "--query-gpu=" + q, "--format=csv,noheader,nounits"]
        bits = [0x8, 0x40, 0x20, 0x4]
        while not self.stop_flag.is_set():
            try:
                r = subprocess.run(cmd, capture_output=True, text=True, timeout=5)
                for ln in r.stdout.splitlines():
                    f = [x.strip() for x in ln.split(",")]
                    if len(f) >= 7:
                        rs = sum(b for b, v in zip(bits, f[3:7]) if v.lower().startswith("active"))
                        self.samples.append((float(f[0]), float(f[1]), float(f[2]), rs))
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def stop(self) -> dict:
        if not self.started:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["not sampled"], "samples": 0}
        self.stop_flag.set()
        self.t.join(timeout=6)
        sm = sorted(x[0] for x in self.samples)
        reasons = set()
        for x in self.samples:
            for bit, name in self.REASONS.items():
                if x[3] & bit:
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max((x[1] for x in self.samples), default=None),
                "power_w_max": max((x[2] for x in self.samples), default=None), "samples": len(sm), "reasons": sorted(reasons),
                "how": self.how}


# ------------------------------------------------------------------------------------------------- reference arm
def cpu_reference_sample(wl: dict, steps: int, warmup: int, t_sample: int = 64):
    """The reference's own algorithm (oracle restatement: one image at a time, encoder once, decoder recomputed over
    the whole prefix each step, probability-product beam scores) on the host cores.  Bounded sample: each step
    captions ONE image with beam `wl['beam']` for `t_sample` decode steps (the full workload decodes 64)."""
    import numpy as np
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import fpnmt_oracle as O
    from fpnmt.weights import init_weights
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    w = init_weights(wl["backbone"], vocab=wl["vocab"], seed=0)
    Wv = O.W(w)
    g = torch.Generator().manual_seed(1234)
    times = []
    for i in range(warmup + steps):
        img = torch.rand(512, 512, 3, generator=g) * 2 - 1
        t0 = time.perf_counter()
        with torch.no_grad():
            O.predict_reference(img, Wv, t_sample, wl["beam"], 2, -1, wl["backbone"], mode="prob")   # end=-1: never stops
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    sec = sum(times) / len(times)
    return dict(value=1.0 / sec, unit="images/s", cores=cores, kind="port",
                sample="1 image of the %d-image batch per step (%s, 512x512), beam=%d, %d of %d decode steps, whole prefix "
                       "recomputed each step (uncached, as utils/pipeline.py:105-112), %d timed steps after %d warm-up, "
                       "PyTorch CPU fp32, %d threads" % (wl["batch"], wl["backbone"], wl["beam"], t_sample, wl["max_len"],
                                                         len(times), warmup, cores),
                sec_per_image=sec)


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = max(1, args.steps)
    warm = max(1, args.warmup)
    cb = cpu_reference_sample(wl, steps, warm)
    line = {"metric": "captioned images/sec", "value": cb["value"], "unit": "images/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": cb["sec_per_image"] * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": wl["name"], "note": "restated reference on host CPU; TensorFlow not installable offline"},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------- own arm
def run_own(args, wl):
    import numpy as np
    import torch
    from fpnmt import dist as fd
    from fpnmt.engine import Engine
    from fpnmt.weights import init_weights

    rank, local, world = fd.init_from_env("nccl")
    if _NCCL_BANNER and rank == 0 and world > 1:
        sys.stderr.write("NCCL version %s\n" % ".".join(str(v) for v in torch.cuda.nccl.version()))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    B, N, V, T = wl["batch"], wl["beam"], wl["vocab"], wl["max_len"]
    w = init_weights(wl["backbone"], vocab=V, seed=0)
    eng_opts = tuple(o for o in args.opts.split(",") if o)
    eng = Engine(w, backbone=wl["backbone"], batch=B, beam=N, vocab=V, max_len=T, precision=args.precision,
                 score_mode="log", use_graphs=not args.no_graphs, device=local, lanes=args.lanes,
                 opts=eng_opts)
    del w
    g = torch.Generator().manual_seed(1234 + rank)
    host_imgs = [(torch.rand(B, 512, 512, 3, generator=g) * 2 - 1).pin_memory() for _ in range(2)]
    dev_imgs = [h.to(dev) for h in host_imgs]
    stream = torch.cuda.current_stream(dev)

    def step_device(i):
        """One-shot call: one batch, nothing else in flight (the latency figure; `one_shot` in the JSON line)."""
        ids, lens = eng.generate(dev_imgs[i % 2], early_stop=False, to_host=False)
        return fd.allgather_captions(ids, lens, world)

    def run_device(n):
        """n whole batches, inputs resident in HBM, through the public streaming call: with lanes >= 2 up to `lanes` batches
        are in flight (fpnmt_submit / fpnmt_collect), so the encoder of batch i+1 runs under the decode of batch i.  Every
        batch is submitted and collected inside the caller's timed region (pipeline fill and drain included)."""
        out = None
        for ids, lens in eng.generate_stream((dev_imgs[i % 2] for i in range(n)), early_stop=False, to_host=False):
            out = fd.allgather_captions(ids, lens, world)
        return out

    def finish_host(ids, lens):
        if world > 1:
            return fd.allgather_captions(ids.to(dev, non_blocking=True), lens.to(dev, non_blocking=True), world)
        return ids, lens

    def run_host_sync(n):
        for i in range(n):
            finish_host(*eng.generate(host_imgs[i % 2], early_stop=False, to_host=True))

    def run_host(n):
        """n whole batches from pinned HOST memory through the public double-buffered call (fpnmt_stage_images +
        fpnmt_generate_staged): n host->device image copies and n device->host result reads, all inside the caller's
        timed region; the copy of batch i+1 overlaps the compute of batch i."""
        for ids, lens in eng.generate_stream((host_imgs[i % 2] for i in range(n)), early_stop=False):
            finish_host(ids, lens)

    for i in range(max(args.warmup, 3)):
        step_device(i)
    # every lane goes through its first use (graph capture + instantiation, pinned staging) before anything is timed
    n_warm = max(args.warmup, 3, 2 * max(1, args.lanes))
    run_device(n_warm)
    torch.cuda.synchronize()
    if args.ncu_step:        # `ncu --profile-from-start off ... bench.py --ncu-step`: capture exactly ONE whole step
        torch.cuda.cudart().cudaProfilerStart()
        step_device(0)
        torch.cuda.synchronize()
        torch.cuda.cudart().cudaProfilerStop()
    # ---- device-resident timing
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    fd.barrier()
    torch.cuda.synchronize()
    l0 = eng.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    out = run_device(args.steps)
    e1.record(stream)
    torch.cuda.synchronize()
    fd.barrier()
    ms = fd.max_over_ranks(e0.elapsed_time(e1), dev)
    launches = eng.launch_count - l0
    clocks = sampler.stop() if rank == 0 else None
    ids_check = out[0].clone()      # the lanes' output buffers are reused by every later call
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ids=out[0], lens=out[1])
    # ---- one batch at a time (nothing else in flight): the latency of a batch, and the cross-check of the lanes' results
    k1 = max(2, min(args.steps, 6))
    fd.barrier()
    torch.cuda.synchronize()
    e0.record(stream)
    for i in range(k1):
        out1 = step_device(args.steps - k1 + i)
    e1.record(stream)
    torch.cuda.synchronize()
    ms_one = fd.max_over_ranks(e0.elapsed_time(e1), dev) / k1
    lanes_equal = bool(torch.equal(out1[0].cpu(), ids_check.cpu()))      # same last batch, one-shot vs streamed through the lanes
    # ... and the latency-optimised configuration: an engine created with lanes = 1 keeps tgemm_kernel (whole weight panel
    # resident, lowest single-chain latency) where lanes >= 2 selects the wide-row Dense kernels built for SM time
    ms_one_l1 = None
    if eng.lanes >= 2 and world == 1 and not args.no_extra:
        eng1 = Engine(init_weights(wl["backbone"], vocab=V, seed=0), backbone=wl["backbone"], batch=B, beam=N, vocab=V, max_len=T,
                      precision=args.precision, score_mode="log", use_graphs=not args.no_graphs, device=local, lanes=1, opts=eng_opts)
        for i in range(3):
            eng1.generate(dev_imgs[i % 2], early_stop=False, to_host=False)
        torch.cuda.synchronize()
        e0.record(stream)
        for i in range(k1):
            eng1.generate(dev_imgs[i % 2], early_stop=False, to_host=False)
        e1.record(stream)
        torch.cuda.synchronize()
        ms_one_l1 = e0.elapsed_time(e1) / k1
        eng1.close()
    # ---- end-to-end timing (host buffers)
    run_host(n_warm)
    torch.cuda.synchronize()
    fd.barrier()
    torch.cuda.synchronize()
    e0.record(stream)
    run_host(args.steps)
    e1.record(stream)
    torch.cuda.synchronize()
    fd.barrier()
    ms_e2e = fd.max_over_ranks(e0.elapsed_time(e1), dev)
    e0.record(stream)
    run_host_sync(args.steps)
    e1.record(stream)
    torch.cuda.synchronize()
    fd.barrier()
    ms_e2e_sync = fd.max_over_ranks(e0.elapsed_time(e1), dev)

    # ---- strong-scaling point (N > 1): the SAME global batch of 64 images cut over the N GPUs (64 / N images per rank)
    strong = None
    if world > 1 and args.workload == "c2" and not args.no_extra and B % world == 0:
        strong = strong_scaling_point(wl, B // world, args, dev, local, world, eng_opts, fd)
    if rank != 0:
        return
    peaks = measured_peaks()
    total_images = B * world * args.steps
    value = total_images / (ms * 1e-3)
    e2e_value = total_images / (ms_e2e * 1e-3)
    # ---- roofline of the dominant kernel, measured live with the engine's per-op CUDA-event profiler
    eng_lanes = eng.lanes
    prof = eng.profile(iters=args.profile_iters)
    if args.profile_out:
        with open(args.profile_out, "w") as f:
            json.dump(prof, f, indent=1)
    # with decoder groups the timed decode runs `decode_groups` concurrent chains over slices of the batch: the launches
    # of one step are those of ONE group's chain (timed alone) times the number of groups
    n_groups = int(prof.get("decode_groups", 1))
    enc_ops = prof["encode"]
    step_ops = prof["decode_group_step"] if n_groups > 1 else prof["decode_step"]
    T_steps = T * n_groups
    # ---- per kernel family: launches per step, device time per step, algorithmic FLOPs / bytes per step
    fam = {}

    def add(ops, mult, family_of):
        for o in ops:
            f = fam.setdefault(family_of(o), dict(launches=0, us=0.0, flops=0.0, bytes=0.0, enc_us=0.0))
            f["launches"] += mult
            f["us"] += o["us"] * mult
            if ops is enc_ops:
                f["enc_us"] += o["us"] * mult
            f["flops"] += o["flops"] * mult
            f["bytes"] += o["bytes"] * mult
    names = {"igemm": "igemm_kernel (tcgen05 implicit-GEMM convolutions / encoder projections)",
             "tgemm": "tgemmw_kernel / tgemm_kernel (tcgen05 Dense layers of the decode step, LayerNorm fused; wide-row kernel when lanes >= 2)",
             "xattn": "xattn_kernel (tcgen05 fused decoder cross-attention block: Q-proj + attention + O-proj + residual + LayerNorm)",
             "dstep": "dstep_kernel (cluster-stationary fused decoder: all layers + vocabulary projection + beam tail of a step, tcgen05)",
             "attention": "attention kernels (mma.sync encoder flash attention; decode self/cross attention)",
             "beam": "k_beam_step (softmax statistics + top-k over beam x vocab + beam bookkeeping)",
             "elementwise": "elementwise NHWC kernels (im2col, pooling, co-attention, LayerNorm, ...)"}
    add(enc_ops, 1, lambda o: o["kind"])
    add(prof.get("decode_init", []), 1, lambda o: o["kind"])
    add(step_ops, T_steps, lambda o: o["kind"])
    total_us = sum(f["us"] for f in fam.values())
    # Share of the TIMED (streamed) step.  With lanes the launches of different batches overlap, so the durations of the launches
    # timed alone no longer add up to the step (the decode chain alone is 64 x ~0.45 ms = 29 ms of a 16 ms step).  The encoder
    # kernels fill the GPU (persistent 148-CTA grids, ~200 KB of shared memory per CTA) and take it exclusively: their time alone is
    # their share of the step; the decode families share what is left of the step in proportion to their time alone.
    step_us = ms / args.steps * 1e3
    enc_total_us = sum(f["enc_us"] for f in fam.values())
    dec_total_us = max(total_us - enc_total_us, 1e-9)
    dec_eff_us = max(step_us - enc_total_us, 0.0) if eng_lanes >= 2 else dec_total_us
    norm = step_us if eng_lanes >= 2 else total_us
    for f in fam.values():
        f["streamed_share"] = (f["enc_us"] + dec_eff_us * (f["us"] - f["enc_us"]) / dec_total_us) / norm
    dom = max(fam, key=lambda k: fam[k]["streamed_share"])
    traffic_tables = {}
    for fn in ("r02_k_ncu_traffic_igemm_encode.json", "r02_k_ncu_traffic_decode_step.json"):
        pth = os.path.join(ROOT, "profiles", fn)
        if os.path.exists(pth):
            with open(pth) as f:
                traffic_tables[fn] = json.load(f)

    def family_entry(k):
        f = fam[k]
        per_launch_us = f["us"] / f["launches"]
        tensor = k in ("igemm", "tgemm", "xattn", "dstep")
        # a kernel timed inside a long step: sustained bf16 peak; HBM peak for the bandwidth-bound families
        peak = peaks["tf_sustained"] if tensor else peaks["hbm_gbs"]
        ach = (f["flops"] / (f["us"] * 1e-6) / 1e12) if tensor else (f["bytes"] / (f["us"] * 1e-6) / 1e9)
        return {"kernel": names.get(k, k), "bound": "tensor" if tensor else "hbm", "achieved": ach, "peak": peak,
                "unit": "TFLOP/s" if tensor else "GB/s", "frac": ach / peak, "launches_per_step": f["launches"],
                "avg_launch_us": per_launch_us, "share_of_step_device_time": f["us"] / total_us,
                "share_of_timed_step": f["streamed_share"],
                "algorithmic_per_launch": (f["flops"] if tensor else f["bytes"]) / f["launches"]}
    roofline = family_entry(dom)
    # measured DRAM traffic per launch of the dominant family (ncu --set full captures summarised under profiles/)
    traffic, traffic_src = None, None
    fam_kernels = {"tgemm": ("tgemm",), "xattn": ("xattn_kernel",), "attention": ("k_dec_self_attention",), "beam": ("k_beam_step",)}
    if dom in fam_kernels and "r02_k_ncu_traffic_decode_step.json" in traffic_tables:
        ks = traffic_tables["r02_k_ncu_traffic_decode_step.json"]["kernels"]
        tg = [v for k, v in ks.items() if k.startswith(fam_kernels[dom])]
        if tg:
            traffic = sum(v["mean_dram_bytes"] * v["launches"] for v in tg) / sum(v["launches"] for v in tg)
            traffic_src = ("profiles/r02_k_ncu_traffic_decode_step.json (ncu --set full of one decode step, mean over its %d %s "
                           "launches, cold cache)" % (sum(v["launches"] for v in tg), dom))
    elif dom == "igemm" and "r02_k_ncu_traffic_igemm_encode.json" in traffic_tables and wl["backbone"] == "resnet50":
        ops_t = traffic_tables["r02_k_ncu_traffic_igemm_encode.json"]["ops"]
        traffic = sum(v["dram_bytes"] for v in ops_t.values()) / len(ops_t)
        traffic_src = ("profiles/r02_k_ncu_traffic_igemm_encode.json (ncu, mean over the %d igemm_kernel launches of one encode)"
                       % len(ops_t))
    roofline["traffic"] = traffic
    roofline["traffic_source"] = traffic_src
    roofline["peak_source"] = peaks["source"] + (", sustained bf16 cuBLAS (kernel timed inside a long step)" if roofline["bound"] == "tensor"
                                                 else ", STREAM-style copy")
    roofline["note"] = ("dominant = kernel family with the largest share of the TIMED step (`share_of_timed_step`): with lanes the "
                        "batches overlap, the encoder kernels (persistent full-GPU grids) keep their time alone and the decode "
                        "families share the rest of the step in proportion to their time alone; `share_of_step_device_time` is the "
                        "share of the sum of all launches timed alone (decode chain un-overlapped).  Live per-op CUDA-event timing by "
                        "fpnmt_profile right after the timed region; `decode_dense` repeats the entry of the decode Dense family")
    if "tgemm" in fam:
        roofline["decode_dense"] = family_entry("tgemm")
    roofline["families"] = {k: family_entry(k) for k in fam}
    ig = [o for o in enc_ops if o["kind"] == "igemm"]
    best = max(ig, key=lambda o: o["flops"] / o["us"])
    roofline["best_tensor_launch"] = {"op": best["name"], "achieved": best["flops"] / (best["us"] * 1e-6) / 1e12, "unit": "TFLOP/s",
                                      "frac_of_burst_peak": best["flops"] / (best["us"] * 1e-6) / 1e12 / peaks["tf"], "us": best["us"]}
    roofline["encode_us_sum"] = sum(o["us"] for o in enc_ops)
    roofline["decode_step_us_sum"] = sum(o["us"] for o in step_ops)
    roofline["decode_step_kernels"] = len(step_ops)
    # ---- fp32-class parity mode (BF16X3: 3-term split-bf16 products, the mode that meets the 2e-3 log-prob / 99 % sequence
    # bound): same workload, same call, device-resident inputs, timed the same way; N = 1 only
    parity_mode = None
    if world == 1 and args.precision == "bf16" and not args.no_parity_mode:
        eng.close()
        w3 = init_weights(wl["backbone"], vocab=V, seed=0)
        eng3 = Engine(w3, backbone=wl["backbone"], batch=B, beam=N, vocab=V, max_len=T, precision="bf16x3", score_mode="log",
                      use_graphs=not args.no_graphs, device=local)
        del w3
        for i in range(3):
            eng3.generate(dev_imgs[i % 2], early_stop=False, to_host=False)
        torch.cuda.synchronize()
        k3 = max(2, min(args.steps, 4))
        e0.record(stream)
        for i in range(k3):
            eng3.generate(dev_imgs[i % 2], early_stop=False, to_host=False)
        e1.record(stream)
        torch.cuda.synchronize()
        ms3 = e0.elapsed_time(e1) / k3
        parity_mode = {"precision": "bf16x3", "value": B / (ms3 * 1e-3), "unit": "images/s", "ms_per_step": ms3, "steps": k3,
                       "note": "same workload in the fp32-class mode whose parity bound is the north star's (log-probs 2e-3, "
                               ">= 99 % identical sequences: tests/test_gpu_captions.py); the headline `value` is the bf16 mode"}
        eng3.close()
    # ---- KV-cache reorder by beam parent as a PHYSICAL move (north-star item 3): same workload with cache_mode="physical";
    # the reorder kernel's achieved HBM bandwidth comes from the per-op profile (CUDA events, algorithmic bytes = 2 x live cache)
    kv_physical = None
    if world == 1 and args.precision == "bf16" and not args.no_parity_mode:
        wp = init_weights(wl["backbone"], vocab=V, seed=0)
        engp = Engine(wp, backbone=wl["backbone"], batch=B, beam=N, vocab=V, max_len=T, precision="bf16", score_mode="log",
                      use_graphs=not args.no_graphs, device=local, cache_mode="physical", decode_path="chain",
                      opts=eng_opts + (("tgemm_wide",) if eng_lanes >= 2 and "no_tgemm_wide" not in eng_opts else ()))   # the kernels of `eng`
        del wp
        for i in range(3):
            ids_p, _ = engp.generate(dev_imgs[i % 2], early_stop=False, to_host=False)
        torch.cuda.synchronize()
        kp = max(2, min(args.steps, 4))
        e0.record(stream)
        for i in range(kp):
            ids_p, _ = engp.generate(dev_imgs[i % 2], early_stop=False, to_host=False)
        e1.record(stream)
        torch.cuda.synchronize()
        msp = e0.elapsed_time(e1) / kp
        ids_p, _ = engp.generate(dev_imgs[(args.steps - 1) % 2], early_stop=False, to_host=False)   # same batch as ids_check
        ids_p = ids_p.clone()                      # before the profiler reuses the engine's buffers
        if not torch.equal(ids_p.cpu(), ids_check.cpu()[:B]):
            sys.stderr.write("physical vs ancestry ids differ: %s %s vs %s %s; rows differing %s; first rows %s | %s\n" % (
                tuple(ids_p.shape), ids_p.dtype, tuple(ids_check.shape), ids_check.dtype,
                int((ids_p.cpu() != ids_check.cpu()[:B]).any(dim=1).sum()) if ids_p.shape == ids_check[:B].shape else "n/a",
                ids_p[0, :8].tolist(), ids_check[0, :8].tolist()))
        profp = engp.profile(iters=args.profile_iters)
        ko = [o for o in profp["decode_step"] if o["kind"] == "kvreorder"]
        gbs = ko[0]["bytes"] / (ko[0]["us"] * 1e-6) / 1e9 if ko else None
        kv_physical = {"value": B / (msp * 1e-3), "unit": "images/s", "ms_per_step": msp, "steps": kp,
                       "kernel": "k_kv_reorder (all layers, K and V, one launch per decode step)",
                       "reorder_us_at_t": ko[0]["us"] if ko else None, "t": profp.get("decode_step_t"),
                       "algorithmic_bytes": ko[0]["bytes"] if ko else None, "achieved_gbs": gbs,
                       "frac_of_hbm_peak": gbs / peaks["hbm_gbs"] if gbs else None,
                       "ids_equal_ancestry_mode": bool(torch.equal(ids_p.cpu(), ids_check.cpu()[:B])),
                       "note": "the default cache mode (ancestry table) moves 4 bytes per (beam, position) instead"}
        engp.close()
    eng.close()
    other = None
    if world == 1 and args.workload == "c2" and args.precision == "bf16" and not args.no_extra:
        other = {k: quick_workload(k, 2, dev, eng_opts) for k in ("c3", "c4")}
    cb = None
    if world == 1 and not args.no_cpu:
        cb = cpu_reference_sample(wl, 3, 1)
        cb = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
    flop_total = B * world * args.steps * (F_ENC[wl["backbone"]] + F_DEC)
    line = {"metric": "captioned images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "bf16x3", "data": "synthetic",
            "config": {"workload": wl["name"], "backbone": wl["backbone"], "batch_per_gpu": B, "beam": N, "vocab": V,
                       "max_len": T, "image": "512x512x3 f32 NHWC", "weights": "random init (Keras default distributions)",
                       "l2": "per-step inputs (%.0f MB) and activations (GBs) exceed the 126 MB L2; two input batches alternate"
                             % (B * 512 * 512 * 3 * 4 / 1e6),
                       "cuda_graphs": not args.no_graphs, "decoder_groups": n_groups, "lanes": eng_lanes,
                       "pipelining": ("%d batches in flight per GPU (fpnmt_submit/fpnmt_collect): encoder of batch i+1 under the "
                                      "decode of batch i; every batch submitted and collected inside the timed region" % eng_lanes)
                                     if eng_lanes > 1 else "none (one batch at a time)",
                       "parallelism": "dp%d (image-sharded, ids all-gather)" % world},
            "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": B * 512 * 512 * 3 * 4,
                    "d2h_bytes_per_step": B * T * 4 + B * 4, "ms_per_step": ms_e2e / args.steps,
                    "api": ("Engine.generate_stream (fpnmt_submit + fpnmt_collect, %d lanes: pinned-host copy, encoder and decode of "
                            "different batches overlap)" % eng_lanes) if eng_lanes > 1 else
                           "Engine.generate_stream (fpnmt_stage_images + fpnmt_generate_staged; double-buffered input)",
                    "unpipelined_value": total_images / (ms_e2e_sync * 1e-3)},
            "one_shot": {"value": B * world / (ms_one * 1e-3), "unit": "images/s", "ms_per_batch": ms_one, "steps": k1,
                         "api": "Engine.generate (one batch, nothing else in flight, device-resident inputs) on the streamed engine",
                         "ids_equal_streamed": lanes_equal,
                         "lanes1_engine": None if ms_one_l1 is None else
                         {"value": B / (ms_one_l1 * 1e-3), "ms_per_batch": ms_one_l1,
                          "note": "Engine(lanes=1): the latency-optimised kernel set (tgemm_kernel) for callers that decode one batch at a time"}},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cb,
            "parity_mode": parity_mode, "kv_cache_physical": kv_physical, "other_workloads": other, "strong_scaling": strong,
            "model_tflops": flop_total / (ms * 1e-3) / 1e12,
            "ids_checksum": int(ids_check.to(torch.int64).sum().item())}
    print(json.dumps(line), flush=True)


def dump_outputs(d, **arrays):
    """DIR/<name>.npy per tensor, as float64 (token ids and lengths are exact in it)."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(d, name + ".npy"), t.cpu().numpy().astype(np.float64))


def quick_workload(key, lanes, dev, opts):
    """Another BASELINE.json config through the same streaming call, device-resident inputs, a short run (driver-visible
    breadth: value, ms per batch and the kernel family with the largest share of the per-op device time)."""
    import torch
    from fpnmt.engine import Engine
    from fpnmt.weights import init_weights
    wl = WORKLOADS[key]
    B, N, V, T = wl["batch"], wl["beam"], wl["vocab"], wl["max_len"]
    eng = Engine(init_weights(wl["backbone"], vocab=V, seed=0), backbone=wl["backbone"], batch=B, beam=N, vocab=V, max_len=T,
                 precision="bf16", score_mode="log", device=dev.index or 0, lanes=lanes, opts=opts)
    g = torch.Generator().manual_seed(99)
    imgs = [(torch.rand(B, 512, 512, 3, generator=g) * 2 - 1).to(dev) for _ in range(2)]

    def run(n):
        for _ in eng.generate_stream((imgs[i % 2] for i in range(n)), early_stop=False, to_host=False):
            pass
    run(2 * lanes)
    torch.cuda.synchronize()
    k = 6
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run(k)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / k
    prof = eng.profile(iters=3)
    fam = {}
    for ops, mult in ((prof["encode"], 1), (prof["decode_step"], T)):
        for o in ops:
            fam[o["kind"]] = fam.get(o["kind"], 0.0) + o["us"] * mult
    eng.close()
    del imgs
    torch.cuda.empty_cache()
    dom = max(fam, key=fam.get)
    return {"workload": wl["name"], "value": B / (ms * 1e-3), "unit": "images/s", "ms_per_step": ms, "steps": k, "lanes": lanes,
            "dominant_family": dom, "dominant_share_of_device_time": fam[dom] / sum(fam.values())}


def strong_scaling_point(wl, b_local, args, dev, local, world, opts, fd):
    """Global batch fixed at the C2 batch (64 images) and cut over the ranks: exposes the latency-bound decode chain that weak
    scaling hides.  Same streaming call, device-resident inputs, max over ranks."""
    import torch
    from fpnmt.engine import Engine
    from fpnmt.weights import init_weights
    N, V, T = wl["beam"], wl["vocab"], wl["max_len"]
    eng = Engine(init_weights(wl["backbone"], vocab=V, seed=0), backbone=wl["backbone"], batch=b_local, beam=N, vocab=V, max_len=T,
                 precision="bf16", score_mode="log", device=local, lanes=args.lanes, opts=opts)
    g = torch.Generator().manual_seed(4321 + local)
    imgs = [(torch.rand(b_local, 512, 512, 3, generator=g) * 2 - 1).to(dev) for _ in range(2)]

    def run(n):
        for ids, lens in eng.generate_stream((imgs[i % 2] for i in range(n)), early_stop=False, to_host=False):
            fd.allgather_captions(ids, lens, world)
    run(2 * max(1, args.lanes))
    fd.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run(args.steps)
    e1.record()
    torch.cuda.synchronize()
    fd.barrier()
    ms = fd.max_over_ranks(e0.elapsed_time(e1), dev)
    eng.close()
    return {"global_batch": b_local * world, "batch_per_gpu": b_local, "value": b_local * world * args.steps / (ms * 1e-3),
            "unit": "images/s", "ms_per_step": ms / args.steps, "steps": args.steps, "scaling": "strong"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="bf16", choices=["bf16", "bf16x3"])
    ap.add_argument("--no-graphs", action="store_true")
    ap.add_argument("--lanes", type=int, default=8, help="batches in flight per GPU (1 = one batch at a time)")
    ap.add_argument("--opts", default="", help="comma-separated fpnmt kernel_opts names (developer A/B, e.g. tgemm_wide)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-parity-mode", action="store_true", help="skip the bf16x3 throughput leg (parity_mode key)")
    ap.add_argument("--no-extra", action="store_true", help="skip the C3 / C4 / strong-scaling legs (other_workloads, strong_scaling keys)")
    ap.add_argument("--profile-iters", type=int, default=10)
    ap.add_argument("--profile-out", default=None, help="write the engine's per-op profile (JSON) here")
    ap.add_argument("--ncu-step", action="store_true", help="bracket one warm step with cudaProfilerStart/Stop (for ncu launch lists)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the token ids and lengths of the last timed step as DIR/ids.npy and DIR/lens.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the CUDA path (--impl own)")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_own(args, wl)
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
