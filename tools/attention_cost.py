"""Time of one Engine.decode_attention call next to Engine.decode_logits at the C2 size (ResNet-50-FPN, batch 64, beam 8,
T = 64, V = 10000, 6 layers, bf16), teacher-forced on T random tokens from the memory of one encode.

    python tools/attention_cost.py [--reps 10] [--out result.json]

Both calls run the same teacher-forced step program T times; decode_attention adds one probability kernel per layer and
step and writes no logits.  CUDA events on the launching stream, the two calls alternated, median over --reps.  The card's
name and power limit are read in the same run and printed with the numbers.

Measured on an NVIDIA B200 at a 1000 W power limit: decode_logits 23.0 ms, decode_attention 29.5 ms (median of 10).
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "fpn-mt-image-captioning_b200"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from fpnmt.engine import Engine
    from fpnmt.weights import init_weights
    B, N, T, V, S = 64, 8, 64, 10000, 512
    eng = Engine(init_weights("resnet50", vocab=V, seed=0), backbone="resnet50", batch=B, beam=N, vocab=V, max_len=T, image_size=S)
    g = torch.Generator(device="cuda").manual_seed(0)
    img = torch.rand((B, S, S, 3), generator=g, device="cuda") * 2 - 1
    mem = eng.encode(img)
    tok = torch.randint(4, V, (B, T), generator=g, device="cuda", dtype=torch.int32)
    tok[:, 0] = 2
    calls = {"decode_logits": lambda: eng.decode_logits(mem, tok), "decode_attention": lambda: eng.decode_attention(mem, tok)}
    for f in calls.values():       # warm-up: module loads, first-touch of the outputs' allocations
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
    res = {"config": "C2 size: resnet50 512x512, batch 64, beam 8, T 64, V 10000, 6 layers, bf16, teacher-forced t = 64",
           "gpu": q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(),
           "median_ms": {k: sorted(v)[len(v) // 2] for k, v in times.items()}, "all_ms": times}
    print(json.dumps(res))
    if args.out:
        json.dump(res, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
