"""Prompted decoding (fpnmt_beam_search_prefix / fpnmt_sample_prefix, include/fpnmt.h) restated on the oracle.  TEST
INFRASTRUCTURE ONLY.

`prefix_beam_search` is the batched KV-cached decode of `diverse_beam_oracle.diverse_beam_search` (G = 1 is the N-best
search, as tests/test_diverse_beam_search.py pins) and `prefix_sample` the decode of `sample_oracle.sample_batch_cached`, each
with the forced step of the definition: at a step t < prefix_len[b] every row of image b takes prefix[b][t], keeps its own
parent, and a live row's score grows by log_softmax(z)[token] (a dead beam stays -inf); nothing is ranked and no draw is
used.  Every other step is the unprompted one, so all prefix_len = 0 reproduces the unprompted oracles exactly.
"""
from __future__ import annotations

from typing import Tuple

import numpy as np
import torch

from fpnmt_oracle.decode import TR, _dec_step_cached, _split_heads, dense, raw_positional_encoding

from beam_search_oracle import length_penalty_table
from diverse_beam_oracle import diverse_step
from sample_oracle import sample_step


def _cross(enc_output, w, N, num_layers, num_heads):
    enc_rows = enc_output.repeat_interleave(N, dim=0)
    cross = []
    for l in range(num_layers):
        p = TR + "/decoder/dec_layers/%d" % l
        cross.append({"k": _split_heads(dense(enc_rows, w, p + "/mha2/wk"), num_heads),
                      "v": _split_heads(dense(enc_rows, w, p + "/mha2/wv"), num_heads)})
    return cross


def forced_step(logits: np.ndarray, score: np.ndarray, fin: np.ndarray, token: int):
    """The forced step of one image: logits (N, V), raw scores (N,).  The score term is diverse_step's raw candidate score."""
    n = logits.shape[0]
    raw = (torch.log_softmax(torch.from_numpy(np.ascontiguousarray(logits, dtype=np.float32)), dim=-1).numpy()
           + score.astype(np.float32)[:, None])
    return np.arange(n), np.full(n, token, np.int64), raw[:, token].astype(np.float32), fin.copy()


def prefix_beam_search(enc_output: torch.Tensor, w, max_seq_len: int, beam: int, beam_groups: int, diversity: float,
                       start: int, end: int, prefix: np.ndarray, prefix_len: np.ndarray, length_penalty: float = 0.0,
                       early_stop: bool = True, num_layers: int = 6, num_heads: int = 8
                       ) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """prefix (B, p) int, prefix_len (B,): valid prefixes (no <end>, ids in range).  Returns ids (B, N, T) int32 (the whole
    caption, prefix included), lens (B, N) and the raw beam scores (B, N) float32, in the output order of
    diverse_beam_search."""
    T, N, G = max_seq_len, beam, beam_groups
    M = N // G
    lp = length_penalty_table(T, length_penalty)
    bsz, _, d = enc_output.shape
    rows = bsz * N
    with torch.no_grad():
        pos = raw_positional_encoding(T, d).to(w.dtype)
        cross = _cross(enc_output, w, N, num_layers, num_heads)
    caches = [{"k": None, "v": None} for _ in range(num_layers)]
    seqs = np.full((bsz, N, 1), start, np.int64)
    score = np.full((bsz, N), -np.inf, np.float32)
    score[:, ::M] = 0.0
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
            if t < prefix_len[b]:
                parent, token, score[b], fin[b] = forced_step(logits[b], score[b], fin[b], int(prefix[b, t]))
            else:
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


def prefix_sample(enc_output: torch.Tensor, w, max_seq_len: int, num_samples: int, start_token: int, end_token: int,
                  prefix: np.ndarray, prefix_len: np.ndarray, temperature: float = 1.0, top_k: int = 0, top_p: float = 1.0,
                  seed: int = 0, num_layers: int = 6, num_heads: int = 8) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """sample_batch_cached with the forced steps: returns ids (B, N, T) int32 (prefix included), lengths (B, N) and fp64
    log-probabilities (B, N), prefix terms included."""
    params = dict(temperature=temperature, top_k=top_k, top_p=top_p, seed=seed)
    bsz, _, d = enc_output.shape
    N, T = num_samples, max_seq_len
    rows = bsz * N
    pos = raw_positional_encoding(T, d).to(w.dtype)
    cross = _cross(enc_output, w, N, num_layers, num_heads)
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
            b = r // N
            if t < prefix_len[b]:
                z = np.asarray(logits[r], np.float64)
                m = z.max()
                token = int(prefix[b, t])
                res = dict(token=token, logprob=float(z[token] - (m + np.log(np.exp(z - m).sum()))))
            else:
                res = sample_step(logits[r], b, r % N, t, params)
            nxt[r] = res["token"]
            if fin[r]:
                continue
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
