"""Developer diagnostic: phase timeline of the fused decoder at the C2 decode shape (needs `build.py --dbg-stamps`).
    FPNMT_DBG_OP=dstep python tests/gpu_diag_timeline.py
"""
import os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "fpn-mt-image-captioning_b200")]
from fpnmt import _lib
_lib.LIB_PATH = os.path.join(ROOT, "fpn-mt-image-captioning_b200", "libfpnmt_dbg.so")
from fpnmt.engine import Engine
from fpnmt.weights import init_weights

def main():
    bb, B, N, V, T = "mobilenet224_1.0", int(os.environ.get("DIAG_B", "64")), 8, 10000, 64
    w = init_weights(bb, vocab=V, seed=0)
    eng = Engine(w, backbone=bb, batch=B, beam=N, vocab=V, max_len=T, decode_path="fused")
    img = (torch.rand(B, 512, 512, 3) * 2 - 1).cuda()
    eng.generate(img, early_stop=False)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    eng.encode(img)
    e0.record()
    ids, lens = eng.decode(early_stop=False, to_host=False)
    e1.record()
    torch.cuda.synchronize()
    print("decode of %d steps: %.3f ms -> %.1f us/step" % (T, e0.elapsed_time(e1), e0.elapsed_time(e1) * 1e3 / T))
    tl = eng.tap("dstep_timeline").cpu().numpy()
    n = int(tl[0]); st = tl[1:1 + n]
    print("steady-state timeline of the last step (us):", " ".join("%.1f" % (x / 1e3) for x in st))
    print("deltas (us):", " ".join("%.1f" % (x / 1e3) for x in np.diff(st)))
    ms = tl[150:174]; ms = ms[ms > 0]
    print("(now: begin, then per group [wait returned, MMAs issued] ...)")
    ps = tl[174:182]
    print("producer: TMA issue time of the 8 ffn1 groups (us since step start):", " ".join("%.2f" % (x / 1e3) for x in ps))
    print("MMA warp, ffn1 job of layer 0 (us since step start): begin, full-wait return of each slot, end:", " ".join("%.2f" % (x / 1e3) for x in ms))
    prof = eng.profile(iters=1)
    print("decode_step op:", [(o["name"][:20], round(o["us"], 1)) for o in prof["decode_step"]], "groups per launch", prof.get("dstep_groups_per_launch"))

if __name__ == "__main__":
    main()
