"""Cost of the N-best and the diverse beam search at the C2 size (ResNet-50-FPN 512x512, batch 64, beam 8, T = 64, V = 10000,
6 layers, bf16, synthetic weights, fixed length).

    python tools/beam_search_cost.py [--reps 10] [--out result.json]

For the default kernels and for opts=("tgemm_wide",) (the logits-free decode tail), on an engine created with true_beam=1,
finished_beams=1 (the beam semantics Engine.beam_search always runs):
1. Engine.beam_search, Engine.beam_search(beam_groups=G, diversity=0.5) for G = 2, 4, 8 and Engine.generate (all from the
   images, early_stop=False, device outputs): CUDA events on the launching stream, the calls alternated, median over --reps.
2. The beam_step op of each: k_beam_step's kernel time from torch.profiler (CUDA activity, mean over the T launches of one
   call of each, in a run of its own after the timed one).  generate runs the <.., false> instantiation, the searches the
   <.., true> one; that one ranks the candidates of each image in G sequential group rankings and writes every beam at the
   close.

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


def beam_step_us(calls):
    from torch.profiler import ProfilerActivity, profile
    out = {}
    for k, f in calls.items():
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            f()
            torch.cuda.synchronize()
        ks = [e for e in prof.events() if "k_beam_step" in e.name and e.device_type == torch.autograd.DeviceType.CUDA]
        us = [e.device_time for e in ks] if ks and hasattr(ks[0], "device_time") else [e.cuda_time for e in ks]
        out[k] = {"kernel": ks[0].name if ks else None, "launches": len(us), "mean_us": sum(us) / max(1, len(us))}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from fpnmt.engine import Engine
    from fpnmt.weights import init_weights
    B, N, T, V, S = 64, 8, 64, 10000, 512
    w = init_weights("resnet50", vocab=V, seed=0)
    g = torch.Generator(device="cuda").manual_seed(0)
    img = torch.rand((B, S, S, 3), generator=g, device="cuda") * 2 - 1
    res = {"config": "C2 size: resnet50 512x512, batch 64, beam 8, T 64, V 10000, 6 layers, bf16, fixed length; engine "
                     "true_beam=1, finished_beams=1"}
    for opts in ((), ("tgemm_wide",)):
        eng = Engine(w, backbone="resnet50", batch=B, beam=N, vocab=V, max_len=T, image_size=S, opts=opts, true_beam=True,
                     finished_beams=True)
        calls = {"generate": lambda: eng.generate(img, early_stop=False, to_host=False),
                 "beam_search": lambda: eng.beam_search(img, early_stop=False, to_host=False, return_logprobs=True)}
        for G in (2, 4, 8):
            calls["diverse_G%d" % G] = (lambda G=G: eng.beam_search(img, early_stop=False, to_host=False, return_logprobs=True,
                                                                     beam_groups=G, diversity=0.5))
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
        res["default" if not opts else "+".join(opts)] = {
            "median_ms": {k: sorted(v)[len(v) // 2] for k, v in times.items()}, "all_ms": times,
            "beam_step_op": beam_step_us(calls)}
        eng.close()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    res["gpu"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()
    print(json.dumps(res))
    if args.out:
        json.dump(res, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
