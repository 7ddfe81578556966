"""Diverse beam search (fpnmt_beam_search_diverse, include/fpnmt.h) restated on the oracle.  TEST INFRASTRUCTURE ONLY.

The beams of a diverse search follow other parents than the plain search's, so this cannot replay the trace of
`predict_batch_cached` the way `beam_search_oracle.beam_search_nbest` does.  `diverse_beam_search` runs its own batched
KV-cached decode on `fpnmt_oracle.decode._dec_step_cached` (the loop of `predict_batch_cached`: cross K/V per row, self-attention
cache reordered by beam parent after every step) and takes each image's step with `diverse_step`, written straight from the
definition: groups ranked in order over their own rows' candidates, every candidate of the row (not only the row's top N),
fp32 keys with one rounding per operation, ties to the lower flat index, then the N-best close with the within-group sort.
"""
from __future__ import annotations

from typing import Tuple

import numpy as np
import torch

from fpnmt_oracle.decode import TR, _dec_step_cached, _split_heads, dense, raw_positional_encoding

from beam_search_oracle import length_penalty_table


def diverse_step(logits: np.ndarray, score: np.ndarray, fin: np.ndarray, lp: np.ndarray, t: int, end: int, groups: int,
                 diversity: float):
    """One step of one image: logits (N, V), score (N,) float32 raw beam scores, fin (N,) 0 = live else the frozen length.
    Returns (parent, token, new raw score, new fin), each (N,), group-major."""
    n, v = logits.shape
    m = n // groups
    raw = (torch.log_softmax(torch.from_numpy(np.ascontiguousarray(logits, dtype=np.float32)), dim=-1).numpy()
           + score.astype(np.float32)[:, None])
    key = np.full((n, v), -np.inf, np.float32)
    for r in range(n):
        if fin[r] > 0:
            raw[r, :] = -np.inf
            raw[r, end] = score[r]                                   # a frozen beam's only candidate is itself
            key[r, end] = np.float32(score[r]) / lp[fin[r]]
        else:
            key[r] = raw[r] / lp[t + 1]
    lam = np.float32(diversity)
    parent = np.zeros(n, np.int64)
    token = np.zeros(n, np.int64)
    h = np.zeros(v, np.int64)                                        # live emissions of each token by earlier groups
    for g in range(groups):
        k = key[g * m:(g + 1) * m].copy()
        for r in range(m):
            if fin[g * m + r] == 0:
                k[r] = k[r] - lam * h.astype(np.float32)             # fp32: one rounding for the product, one for the difference
        order = np.argsort(-k.reshape(-1), kind="stable")[:m]         # ties -> lower flat index within the group
        parent[g * m:(g + 1) * m] = g * m + order // v
        token[g * m:(g + 1) * m] = order % v
        for p, tk in zip(parent[g * m:(g + 1) * m], token[g * m:(g + 1) * m]):
            if fin[p] == 0:
                h[tk] += 1
    new_fin = np.where(fin[parent] > 0, fin[parent], np.where(token == end, t + 1, 0))
    return parent, token, raw[parent, token].astype(np.float32), new_fin


def diverse_beam_search(enc_output: torch.Tensor, w, max_seq_len: int, beam: int, beam_groups: int, diversity: float,
                        start: int, end: int, length_penalty: float = 0.0, early_stop: bool = True, num_layers: int = 6,
                        num_heads: int = 8) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Returns ids (B, N, T) int32 (no <start>, no <end>, 0 from len on), lens (B, N) int32 (T: truncated) and the raw beam
    scores (B, N) float32, group-major and sorted within each group by score / lp(min(len + 1, T)) (ties: lower slot).
    early_stop=False closes every image at the last step instead of at the step where its last beam froze, and decodes
    all T steps (the result must be the same)."""
    T, N, G = max_seq_len, beam, beam_groups
    M = N // G
    lp = length_penalty_table(T, length_penalty)
    bsz, _, d = enc_output.shape
    rows = bsz * N
    with torch.no_grad():
        enc_rows = enc_output.repeat_interleave(N, dim=0)
        pos = raw_positional_encoding(T, d).to(w.dtype)
        cross = []
        for l in range(num_layers):
            p = TR + "/decoder/dec_layers/%d" % l
            cross.append({"k": _split_heads(dense(enc_rows, w, p + "/mha2/wk"), num_heads),
                          "v": _split_heads(dense(enc_rows, w, p + "/mha2/wv"), num_heads)})
    caches = [{"k": None, "v": None} for _ in range(num_layers)]
    seqs = np.full((bsz, N, 1), start, np.int64)
    score = np.full((bsz, N), -np.inf, np.float32)
    score[:, ::M] = 0.0                                              # the first beam of every group
    fin = np.zeros((bsz, N), np.int64)
    done = np.zeros(bsz, bool)
    ids = np.zeros((bsz, N, T), np.int32)
    lens = np.zeros((bsz, N), np.int32)
    logprob = np.zeros((bsz, N), np.float32)
    for t in range(T):
        with torch.no_grad():
            tok = torch.from_numpy(seqs[:, :, -1].reshape(rows))
            logits = _dec_step_cached(w, tok, pos[t], caches, cross, num_layers, num_heads).to(torch.float32).numpy()
        logits = logits.reshape(bsz, N, -1)
        gparent = np.zeros((bsz, N), np.int64)
        new_seqs = np.zeros((bsz, N, t + 2), np.int64)
        for b in range(bsz):
            parent, token, score[b], fin[b] = diverse_step(logits[b], score[b], fin[b], lp, t, end, G, diversity)
            gparent[b] = b * N + parent
            new_seqs[b] = np.concatenate([seqs[b][parent], token[:, None]], axis=-1)
        seqs = new_seqs
        gp = torch.from_numpy(gparent.reshape(rows))
        for c in caches:
            c["k"], c["v"] = c["k"][gp], c["v"][gp]
        for b in range(bsz):
            if done[b] or not ((early_stop and (fin[b] > 0).all()) or t == T - 1):
                continue
            ln = np.where(fin[b] > 0, fin[b] - 1, t + 1)
            key = score[b] / lp[np.minimum(ln + 1, T)]
            for g in range(G):
                order = g * M + np.argsort(-key[g * M:(g + 1) * M], kind="stable")
                for slot, n in zip(range(g * M, (g + 1) * M), order):
                    ids[b, slot, :ln[n]] = seqs[b, n, 1:1 + ln[n]]
                    lens[b, slot] = ln[n]
                    logprob[b, slot] = score[b, n]
            done[b] = True
        if early_stop and done.all():
            break
    return ids, lens, logprob
