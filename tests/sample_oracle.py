"""fp64 restatement of sampled caption decoding (fpnmt_sampling, include/fpnmt.h).  TEST INFRASTRUCTURE ONLY.

`philox4x32_10` is the counter-based generator in integer numpy; `sample_step` is one step of one row, implemented
literally from the header's definition with a sort (no fixed point, no radix select); `sample_batch_cached` runs the
KV-cached oracle decoder (`fpnmt_oracle.decode._dec_step_cached`) with every row an independent sample and no cache reorder.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import numpy as np
import torch

from fpnmt_oracle.decode import _dec_step_cached, _split_heads
from fpnmt_oracle.model import TR, dense, raw_positional_encoding

_M0, _M1, _W0, _W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
_MASK = 0xFFFFFFFF


def philox4x32_10(counter, key) -> np.ndarray:
    """Philox4x32-10 (Salmon et al., SC'11): counter (4,) and key (2,) uint32 -> (4,) uint32.  Leading batch dimensions
    broadcast."""
    c = [np.asarray(x, np.uint64) & _MASK for x in np.moveaxis(np.asarray(counter, np.uint64), -1, 0)]
    k = [np.asarray(x, np.uint64) & _MASK for x in np.moveaxis(np.asarray(key, np.uint64), -1, 0)]
    for r in range(10):
        if r:
            k = [(k[0] + _W0) & _MASK, (k[1] + _W1) & _MASK]
        p0 = np.uint64(_M0) * c[0]
        p1 = np.uint64(_M1) * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & _MASK
        hi1, lo1 = p1 >> np.uint64(32), p1 & _MASK
        c = [hi1 ^ c[1] ^ k[0], lo1, hi0 ^ c[3] ^ k[1], lo0]
    return np.stack(c, -1).astype(np.uint32)


def uniform(t: int, b: int, n: int, seed: int) -> float:
    """u = (philox(counter = (t, b, n, 0), key = (seed lo, seed hi))[0] >> 8) * 2^-24 (exact in fp32 and fp64)."""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    r = philox4x32_10([t, b, n, 0], [seed & _MASK, seed >> 32])
    return float(int(r[0]) >> 8) * 2.0 ** -24


def sample_step(logits, b: int, n: int, t: int, params: Dict) -> Dict:
    """One row.  params: temperature, top_k, top_p, seed.  Returns token, logprob (log_softmax at temperature 1), u, the sets
    K1 and K2 (boolean masks), the renormalised distribution over K2 (`q`) and `margin`: the distance, as a fraction of K2's
    mass (CDF) or of K1's mass (nucleus), from u * mass to the nearest CDF step and from the nucleus target to the nearest
    cumulative mass at which K2 would change - a row with a small margin may legitimately draw differently in fp32."""
    z = np.asarray(logits, np.float64)
    V = z.shape[0]
    T_, k, p_top = float(params.get("temperature", 1.0)), int(params.get("top_k", 0)), float(params.get("top_p", 1.0))
    m = z.max()
    lse = m + np.log(np.exp(z - m).sum())
    u = uniform(t, b, n, params.get("seed", 0))
    if T_ == 0.0:
        tok = int(np.argmax(z))                             # lowest id among the maxima
        K = z == z[tok]
        return dict(token=tok, logprob=float(z[tok] - lse), u=u, K1=K, K2=K, q=K / K.sum(), margin=np.inf)
    K1 = np.ones(V, bool)
    if 0 < k < V:
        zk = np.sort(z)[::-1][k - 1]
        K1 = z >= zk
    p = np.where(K1, np.exp((z - m) / T_), 0.0)
    p = p / p.sum()
    K2 = K1.copy()
    margin = np.inf
    if p_top < 1.0:
        ps = np.sort(p[K1])[::-1]
        cum = np.cumsum(ps)
        target = p_top * cum[-1]
        j = int(np.argmax(cum >= target))                   # first prefix reaching the target
        tau = ps[j]
        K2 = K1 & (p >= tau)
        # cumulative masses at the ends of the distinct-value groups around the cut
        ends = np.flatnonzero(np.r_[ps[1:] != ps[:-1], True])
        cums = cum[ends]
        margin = float(np.min(np.abs(cums - target)) / cum[-1])
    w = np.where(K2, p, 0.0)
    c = np.cumsum(w)
    S = c[-1]
    tok = int(np.argmax(c > u * S))
    steps = c[K2]
    margin = min(margin, float(np.min(np.abs(np.r_[0.0, steps] - u * S)) / S))
    return dict(token=tok, logprob=float(z[tok] - lse), u=u, K1=K1, K2=K2, q=w / S, margin=margin)


def sample_batch_cached(enc_output: torch.Tensor, w, max_seq_len: int, num_samples: int, start_token: int, end_token: int,
                        temperature: float = 1.0, top_k: int = 0, top_p: float = 1.0, seed: int = 0, num_layers: int = 6,
                        num_heads: int = 8, trace: Optional[dict] = None) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """num_samples independent sampled captions per image from the KV-cached decoder (rows never reordered).

    Returns ids (B, N, T) int32 zero padded (no <start>, no <end>), lengths (B, N) int32 (T when <end> never fired) and
    log-probabilities (B, N) float64: the sum of log_softmax(z)[token] at temperature 1 over the emitted steps, <end>
    included.  A finished sample's row keeps being computed; its tokens are ignored.  trace["margin"] collects the
    `sample_step` margins of every draw that entered a caption, trace["top2_gap"] the gaps between the two largest logits
    of those rows (0: an exact top-1 tie)."""
    params = dict(temperature=temperature, top_k=top_k, top_p=top_p, seed=seed)
    bsz, _, d = enc_output.shape
    N, T = num_samples, max_seq_len
    rows = bsz * N
    enc_rows = enc_output.repeat_interleave(N, dim=0)
    pos = raw_positional_encoding(T, d).to(w.dtype)
    cross = []
    for l in range(num_layers):
        p = TR + "/decoder/dec_layers/%d" % l
        cross.append({"k": _split_heads(dense(enc_rows, w, p + "/mha2/wk"), num_heads),
                      "v": _split_heads(dense(enc_rows, w, p + "/mha2/wv"), num_heads)})
    caches = [{"k": None, "v": None} for _ in range(num_layers)]
    tok = np.full((rows,), start_token, np.int64)
    fin = np.zeros((rows,), bool)
    ids = np.zeros((rows, T), np.int32)
    lens = np.zeros((rows,), np.int32)
    lp = np.zeros((rows,), np.float64)
    for t in range(T):
        with torch.no_grad():
            logits = _dec_step_cached(w, torch.from_numpy(tok), pos[t], caches, cross, num_layers, num_heads)
        logits = logits.to(torch.float32).numpy()
        nxt = np.zeros_like(tok)
        for r in range(rows):
            res = sample_step(logits[r], r // N, r % N, t, params)
            nxt[r] = res["token"]
            if fin[r]:
                continue
            if trace is not None:
                trace.setdefault("margin", []).append(res["margin"])
                top2 = np.sort(logits[r])[-2:]
                trace.setdefault("top2_gap", []).append(float(top2[1] - top2[0]))
            lp[r] += res["logprob"]
            if res["token"] == end_token:
                fin[r] = True
            else:
                ids[r, lens[r]] = res["token"]
                lens[r] += 1
                if t == T - 1:
                    fin[r] = True
        tok = nxt
        if fin.all():
            break
    return ids.reshape(bsz, N, T), lens.reshape(bsz, N), lp.reshape(bsz, N)
