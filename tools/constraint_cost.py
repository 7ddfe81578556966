"""Cost of constrained decoding at the C2 size (ResNet-50-FPN 512x512, batch 64, beam 8, T = 64, V = 10000, 6 layers, bf16,
synthetic weights, fixed length).

    python tools/constraint_cost.py [--reps 7] [--out result.json]

For the default kernels and for opts=("tgemm_wide",) (the logits-free decode tail):
1. Engine.beam_search and Engine.sample unconstrained and constrained (no_repeat_ngram 3, min_len 5, 3 banned ids; all from
   the images, early_stop=False, device outputs): CUDA events on the launching stream, the calls alternated, median over
   --reps.  A constrained call runs the same steps plus the ban-set reads and writes (under 1 MB per step at this size).
2. In a run of its own, the vocabulary projection of the logits-free tail at the C2 shape (512 rows, K 512, V 10000) through
   the stand-alone operators: tgemmw_target_kernel (fpnmt_op_vocab_stats_target, the prompted search) against
   tgemmw_mask_kernel (fpnmt_op_vocab_stats_mask with a target, the constrained search), kernel time from torch.profiler
   (CUDA activity, mean over 50 launches of each, alternated).

The card's name and power limit are read in the same run and printed with the numbers.  Measured on one NVIDIA B200 at a
1000 W power limit (--reps 7): beam_search 29.41 ms, constrained 29.77 ms; sample 45.49 ms, constrained 45.94 ms; with
tgemm_wide beam_search 35.47 ms, constrained 36.25 ms, sample 51.62 ms, constrained 52.08 ms; the projection alone 35.0 us
(tgemmw_target_kernel) against 37.8 us (tgemmw_mask_kernel).
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "fpn-mt-image-captioning_b200"))

CONSTRAINTS = dict(no_repeat_ngram=3, min_len=5, banned=[0, 1, 2])


def final_layer_us(reps=50):
    import numpy as np
    from torch.profiler import ProfilerActivity, profile
    from fpnmt.engine import vocab_stats_mask, vocab_stats_target
    R, K, F = 512, 512, 10000
    rng = np.random.default_rng(0)
    x = torch.from_numpy(rng.standard_normal((R, K)).astype(np.float32)).cuda()
    kern = (rng.standard_normal((K, F)) / np.sqrt(K)).astype(np.float32)
    bias = (rng.standard_normal(F) * 0.1).astype(np.float32)
    tgt = torch.from_numpy(rng.integers(0, F, R).astype(np.int32)).cuda()
    ban = np.zeros((R, (F + 31) // 32), np.uint32)                  # 3 static ids + 3 repeat bans per row
    for v in list(CONSTRAINTS["banned"]) + list(rng.integers(0, F, 3)):
        ban[:, v // 32] |= np.uint32(1 << (v % 32))
    mask = torch.from_numpy(ban.view(np.int32)).cuda()
    vocab_stats_target(x, kern, tgt, bias)
    vocab_stats_mask(x, kern, mask, bias, target=tgt)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            vocab_stats_target(x, kern, tgt, bias)
            vocab_stats_mask(x, kern, mask, bias, target=tgt)
        torch.cuda.synchronize()
    out = {}
    for n in ("tgemmw_target_kernel", "tgemmw_mask_kernel"):
        ks = [e for e in prof.events() if n + "(" in e.name and e.device_type == torch.autograd.DeviceType.CUDA]
        us = [e.device_time for e in ks] if ks and hasattr(ks[0], "device_time") else [e.cuda_time for e in ks]
        out[n] = {"launches": len(us), "mean_us": sum(us) / max(1, len(us)), "median_us": sorted(us)[len(us) // 2] if us else None}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from fpnmt.engine import Engine
    from fpnmt.weights import init_weights
    B, N, T, V, S = 64, 8, 64, 10000, 512
    w = init_weights("resnet50", vocab=V, seed=0)
    g = torch.Generator(device="cuda").manual_seed(0)
    img = torch.rand((B, S, S, 3), generator=g, device="cuda") * 2 - 1
    res = {"config": "C2 size: resnet50 512x512, batch 64, beam 8, T 64, V 10000, 6 layers, bf16, fixed length; constraints "
                     "no_repeat_ngram 3, min_len 5, banned ids 0, 1, 2"}
    for opts in ((), ("tgemm_wide",)):
        eng = Engine(w, backbone="resnet50", batch=B, beam=N, vocab=V, max_len=T, image_size=S, opts=opts)
        kw = dict(early_stop=False, to_host=False, return_logprobs=True)
        sp = dict(temperature=0.9, top_k=50, top_p=0.95, seed=1)
        calls = {"beam_search": lambda: eng.beam_search(img, **kw),
                 "beam_search_constrained": lambda: eng.beam_search(img, **kw, **CONSTRAINTS),
                 "sample": lambda: eng.sample(img, **kw, **sp),
                 "sample_constrained": lambda: eng.sample(img, **kw, **sp, **CONSTRAINTS)}
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
        res["default" if not opts else "+".join(opts)] = {"median_ms": {k: sorted(v)[len(v) // 2] for k, v in times.items()},
                                                          "all_ms": times}
        eng.close()
    res["final_layer_C2_shape"] = final_layer_us()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    res["gpu"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()
    print(json.dumps(res))
    if args.out:
        json.dump(res, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
