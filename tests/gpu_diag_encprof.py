"""Diagnostic: per-op encode profile of the C2 encoder for a few layers (A/B of kernel_opts via DIAG_OPTS)."""
import os, sys, json
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "fpn-mt-image-captioning_b200"))
import torch
from fpnmt.engine import Engine
from fpnmt.weights import init_weights
w = init_weights("resnet50", vocab=1000, seed=0)
eng = Engine(w, backbone="resnet50", batch=64, beam=8, vocab=1000, max_len=4, opts=tuple(o for o in os.environ.get("DIAG_OPTS", "").split(",") if o))
img = torch.rand(64, 512, 512, 3).cuda() * 2 - 1
eng.generate(img, early_stop=False)
p = eng.profile(iters=5)
names = ("res2a_2c", "res2a_1", "res3a_2c", "res2a_2a", "res4a_2c", "enc_kv_view0", "res2a_2b", "P3_trunk0")
print(os.environ.get("DIAG_OPTS"), round(sum(o["us"] for o in p["encode"])), [(o["name"], round(o["us"], 1)) for o in p["encode"] if o["name"] in names])
