"""Time of Engine.score at the C2 size (ResNet-50-FPN, batch 64, N = 8 captions per image, t = 64, V = 10000, 6 layers,
bf16) next to the slow way to the same numbers: N sequential decode_logits calls (the KV-cached step program, t steps each)
followed by torch log_softmax and gather.

    python tools/score_cost.py [--reps 10] [--out result.json]

The two whole calls alternate (CUDA events on the launching stream, median over --reps, memory of one encode, random
caption ids and lengths).  Then one score call runs under torch.profiler (a pass of its own) for the device time of the
new kernels per call: the causal self-attention (all 6 layers) and score_rows (all t chunks).  The device memory the first
score call allocates (activations for B * N * max_len rows and the per-row buffers) is read with cudaMemGetInfo.  The
card's name and power limit are read in the same run and printed with the numbers.

Measured on an NVIDIA B200 at a 1000 W power limit (median of 10): score 8.30 ms, decode_logits x 8 with log_softmax and
gather 185.6 ms (22x).  Device time per score call: k_score_self_attention 2.74 ms (6 layers), k_score_rows 1.39 ms (64
chunks), k_score_embed 0.04 ms, k_score_sum 0.03 ms.  The first call allocates 448 MB.  Largest difference of a caption's
total between the two paths: 0.46 (bf16, up to 65 terms per caption).
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
    ids = torch.randint(4, V, (B, N, T), generator=g, device="cuda", dtype=torch.int32)
    lens = torch.randint(8, T + 1, (B, N), generator=g, device="cuda", dtype=torch.int32)
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    eng.score(ids, lens, to_host=False)
    torch.cuda.synchronize()
    score_bytes = free0 - torch.cuda.mem_get_info()[0]

    def slow():
        out = torch.zeros((B, N), device="cuda")
        for n in range(N):
            tok = torch.cat([torch.full((B, 1), 2, dtype=torch.int32, device="cuda"), ids[:, n, :T - 1]], 1)
            lsm = torch.log_softmax(eng.decode_logits(mem, tok), -1)
            tgt = ids[:, n].long().clone()
            tgt.scatter_(1, lens[:, n:n + 1].long().clamp(max=T - 1), 3)
            terms = lsm.gather(2, tgt[..., None])[..., 0]
            n_bn = torch.where(lens[:, n] < T, lens[:, n] + 1, T)
            out[:, n] = (terms * (torch.arange(T, device="cuda")[None] < n_bn[:, None])).sum(1)
        return out

    calls = {"score": lambda: eng.score(ids, lens, to_host=False), "decode_logits_x_N": slow}
    for f in calls.values():       # warm-up: module loads, graph capture, first-touch of the outputs' allocations
        f()
    torch.cuda.synchronize()
    fast_lp, slow_lp = calls["score"](), slow()
    max_diff = float((fast_lp - slow_lp).abs().max())
    times = {k: [] for k in calls}
    for _ in range(args.reps):
        for k, f in calls.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1))
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.score(ids, lens, to_host=False)
        torch.cuda.synchronize()
    kern = {}
    for e in prof.key_averages():
        for key in ("k_score_self_attention", "k_score_rows", "k_score_embed", "k_score_sum"):
            if key in e.key:
                dt = getattr(e, "device_time_total", None)
                if dt is None:
                    dt = e.cuda_time_total
                kern[key] = kern.get(key, 0.0) + dt / 1000.0
    eng.close()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    res = {"config": "C2 size: resnet50 512x512, batch 64, N 8 captions per image, t 64, V 10000, 6 layers, bf16",
           "gpu": q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(),
           "median_ms": {k: sorted(v)[len(v) // 2] for k, v in times.items()}, "all_ms": times,
           "kernel_ms_per_score_call": kern, "score_alloc_MB": score_bytes / 2**20,
           "max_abs_diff_total_logprob_vs_slow": max_diff}
    print(json.dumps(res))
    if args.out:
        json.dump(res, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
