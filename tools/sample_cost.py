"""Cost of sampled decoding at the C2 size (ResNet-50-FPN 512x512, batch 64, beam 8 = 8 samples per image, T = 64,
V = 10000, 6 layers, bf16).

    python tools/sample_cost.py [--reps 10] [--out result.json]

1. k_sample_step alone on [512][10000] fp32 logits (20.5 MB read per call), through fpnmt_op_sample_step, for greedy, plain,
   top-k + top-p and top-p-only parameters: kernel time from torch.profiler (CUDA activity of k_sample_step, mean over the
   calls).  Eight logits buffers (164 MB, more than the 126 MB L2) are used in turn, so every call reads its row from HBM.
   Printed next to the HBM floor of the bytes at 6.54 TB/s.
2. Engine.sample against Engine.generate (both fixed length, T steps, from the images, device outputs): CUDA events on the
   launching stream, the two calls alternated, median over --reps.

The card's name and power limit are read in the same run and printed with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "fpn-mt-image-captioning_b200"))


def kernel_times(rows, V, reps):
    from torch.profiler import ProfilerActivity, profile
    from fpnmt.engine import sample_step
    g = torch.Generator(device="cuda").manual_seed(1)
    bufs = [torch.randn((rows, V), generator=g, device="cuda") * 3 for _ in range(8)]
    cases = {"greedy": dict(temperature=0.0), "plain": dict(temperature=1.0),
             "top_k20_top_p0.95": dict(temperature=0.8, top_k=20, top_p=0.95), "top_p0.9": dict(temperature=1.0, top_p=0.9)}
    out = {}
    for name, kw in cases.items():
        for i in range(3):
            sample_step(bufs[i], 8, i, seed=i, **kw)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(reps):
                sample_step(bufs[i % 8], 8, i, seed=i, **kw)
            torch.cuda.synchronize()
        ks = [e for e in prof.events() if "k_sample_step" in e.name and e.device_type == torch.autograd.DeviceType.CUDA]
        us = [e.device_time for e in ks] if ks and hasattr(ks[0], "device_time") else [e.cuda_time for e in ks]
        out[name] = {"calls": len(us), "mean_us": sum(us) / max(1, len(us)), "min_us": min(us) if us else None}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from fpnmt.engine import Engine
    from fpnmt.weights import init_weights
    B, N, T, V, S = 64, 8, 64, 10000, 512
    rows = B * N
    bytes_ = rows * V * 4
    kern = kernel_times(rows, V, 40)
    eng = Engine(init_weights("resnet50", vocab=V, seed=0), backbone="resnet50", batch=B, beam=N, vocab=V, max_len=T, image_size=S)
    g = torch.Generator(device="cuda").manual_seed(0)
    img = torch.rand((B, S, S, 3), generator=g, device="cuda") * 2 - 1
    calls = {"generate": lambda: eng.generate(img, early_stop=False, to_host=False),
             "sample": lambda: eng.sample(img, temperature=0.8, top_k=20, top_p=0.95, seed=1, early_stop=False, to_host=False)}
    for f in calls.values():       # warm-up: module loads, graph capture, first-touch of the buffers
        f()
    torch.cuda.synchronize()
    times = {k: [] for k in calls}
    for _ in range(args.reps):
        for k, f in calls.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1))
    eng.close()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    res = {"config": "C2 size: resnet50 512x512, batch 64, beam 8, T 64, V 10000, 6 layers, bf16, fixed length",
           "gpu": q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(),
           "k_sample_step": {"rows": rows, "V": V, "bytes": bytes_, "hbm_floor_us_at_6.54TBps": bytes_ / 6.54e12 * 1e6,
                             "cases": kern},
           "median_ms": {k: sorted(v)[len(v) // 2] for k, v in times.items()}, "all_ms": times}
    print(json.dumps(res))
    if args.out:
        json.dump(res, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
