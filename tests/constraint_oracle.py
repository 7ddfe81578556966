"""Constrained decoding (fpnmt_beam_search_constrained / fpnmt_sample_constrained, include/fpnmt.h) restated on the oracle.
TEST INFRASTRUCTURE ONLY.

`ban_set` is the definition of a row's ban set A(t) = S | E(t) | R(t).  `constrained_beam_search` is the KV-cached decode of
prefix_oracle.prefix_beam_search whose free step is `constrained_diverse_step`: diverse_beam_oracle.diverse_step with the
ranking key of a live row at -inf on its ban set (raw scores still from the unmasked log_softmax).  `constrained_sample` is
prefix_oracle.prefix_sample whose free step is `constrained_sample_step`: sample_oracle.sample_step on z with the banned
logits at -inf, reporting log_softmax of the unmasked z.  Forced prefix steps ignore the ban set.  With no constraint both
reproduce the prefix oracles exactly.
"""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from fpnmt_oracle.decode import _dec_step_cached, raw_positional_encoding

from beam_search_oracle import length_penalty_table
from prefix_oracle import _cross, forced_step
from sample_oracle import sample_step


def ban_set(caption: Sequence[int], V: int, end: int, no_repeat_ngram: int = 0, min_len: int = 0,
            banned: Optional[Sequence[int]] = None) -> np.ndarray:
    """A(t) of a row whose caption so far (no <start>, prefix included) is `caption`, t = len(caption): boolean (V,)."""
    w = [int(x) for x in caption]
    t, n = len(w), int(no_repeat_ngram)
    a = np.zeros(V, bool)
    if banned is not None and len(banned):
        a[np.asarray(banned, np.int64)] = True
    if t < min_len:
        a[end] = True
    if n >= 1:
        tail = w[t - n + 1:] if n > 1 else []
        for j in range(0, t - n + 1):
            if w[j:j + n - 1] == tail:
                a[w[j + n - 1]] = True
    return a


def constrained_diverse_step(logits: np.ndarray, score: np.ndarray, fin: np.ndarray, lp: np.ndarray, t: int, end: int,
                             groups: int, diversity: float, ban: np.ndarray):
    """diverse_step of one image with ban (N, V) bool: a live row's banned candidates are never ranked."""
    n, v = logits.shape
    m = n // groups
    raw = (torch.log_softmax(torch.from_numpy(np.ascontiguousarray(logits, dtype=np.float32)), dim=-1).numpy()
           + score.astype(np.float32)[:, None])
    key = np.full((n, v), -np.inf, np.float32)
    for r in range(n):
        if fin[r] > 0:
            raw[r, :] = -np.inf
            raw[r, end] = score[r]
            key[r, end] = np.float32(score[r]) / lp[fin[r]]
        else:
            key[r] = np.where(ban[r], np.float32(-np.inf), raw[r] / lp[t + 1])
    lam = np.float32(diversity)
    parent = np.zeros(n, np.int64)
    token = np.zeros(n, np.int64)
    h = np.zeros(v, np.int64)
    for g in range(groups):
        k = key[g * m:(g + 1) * m].copy()
        for r in range(m):
            if fin[g * m + r] == 0:
                k[r] = k[r] - lam * h.astype(np.float32)
        order = np.argsort(-k.reshape(-1), kind="stable")[:m]
        parent[g * m:(g + 1) * m] = g * m + order // v
        token[g * m:(g + 1) * m] = order % v
        for p, tk in zip(parent[g * m:(g + 1) * m], token[g * m:(g + 1) * m]):
            if fin[p] == 0:
                h[tk] += 1
    new_fin = np.where(fin[parent] > 0, fin[parent], np.where(token == end, t + 1, 0))
    return parent, token, raw[parent, token].astype(np.float32), new_fin


def constrained_sample_step(logits, b: int, n: int, t: int, params, ban: np.ndarray):
    """sample_step on the masked z (selection only); logprob = log_softmax of the unmasked z."""
    z = np.asarray(logits, np.float64)
    res = sample_step(np.where(ban, -np.inf, z), b, n, t, params)
    m = z.max()
    res["logprob"] = float(z[res["token"]] - (m + np.log(np.exp(z - m).sum())))
    return res


def constrained_beam_search(enc_output: torch.Tensor, w, max_seq_len: int, beam: int, beam_groups: int, diversity: float,
                            start: int, end: int, no_repeat_ngram: int = 0, min_len: int = 0, banned=None,
                            prefix: Optional[np.ndarray] = None, prefix_len: Optional[np.ndarray] = None,
                            length_penalty: float = 0.0, early_stop: bool = True, num_layers: int = 6, num_heads: int = 8
                            ) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """prefix_beam_search with the constraints; prefix None = unprompted.  Returns ids (B, N, T), lens (B, N), raw scores."""
    T, N, G = max_seq_len, beam, beam_groups
    M = N // G
    lp = length_penalty_table(T, length_penalty)
    bsz, _, d = enc_output.shape
    rows = bsz * N
    if prefix is None:
        prefix, prefix_len = np.zeros((bsz, 1), np.int32), np.zeros(bsz, np.int32)
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
        V = logits.shape[-1]
        gparent = np.zeros((bsz, N), np.int64)
        new_seqs = np.zeros((bsz, N, t + 2), np.int64)
        for b in range(bsz):
            if t < prefix_len[b]:
                parent, token, score[b], fin[b] = forced_step(logits[b], score[b], fin[b], int(prefix[b, t]))
            else:
                ban = np.stack([ban_set(seqs[b, r, 1:], V, end, no_repeat_ngram, min_len, banned) for r in range(N)])
                parent, token, score[b], fin[b] = constrained_diverse_step(logits[b], score[b], fin[b], lp, t, end, G,
                                                                           diversity, ban)
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


def constrained_sample(enc_output: torch.Tensor, w, max_seq_len: int, num_samples: int, start_token: int, end_token: int,
                       no_repeat_ngram: int = 0, min_len: int = 0, banned=None, prefix: Optional[np.ndarray] = None,
                       prefix_len: Optional[np.ndarray] = None, temperature: float = 1.0, top_k: int = 0, top_p: float = 1.0,
                       seed: int = 0, num_layers: int = 6, num_heads: int = 8) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """prefix_sample with the constraints; prefix None = unprompted.  Returns ids (B, N, T), lengths and fp64 logprobs."""
    params = dict(temperature=temperature, top_k=top_k, top_p=top_p, seed=seed)
    bsz, _, d = enc_output.shape
    N, T = num_samples, max_seq_len
    rows = bsz * N
    if prefix is None:
        prefix, prefix_len = np.zeros((bsz, 1), np.int32), np.zeros(bsz, np.int32)
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
        V = logits.shape[-1]
        nxt = np.zeros_like(tok)
        for r in range(rows):
            b = r // N
            if t < prefix_len[b]:
                z = np.asarray(logits[r], np.float64)
                m = z.max()
                token = int(prefix[b, t])
                res = dict(token=token, logprob=float(z[token] - (m + np.log(np.exp(z - m).sum()))))
            else:
                ban = ban_set(ids[r, :lens[r]], V, end_token, no_repeat_ngram, min_len, banned)
                res = constrained_sample_step(logits[r], b, r % N, t, params, ban)
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


def check_caption(cap: Sequence[int], no_repeat_ngram: int, min_len: int, banned, prefix_len: int) -> None:
    """The structural guarantees of one returned caption (asserts): no banned id after the prefix, no n-gram ending at a
    position >= prefix_len that also occurs earlier, and at least min_len tokens (<end> is banned before that, and a caption
    that never ends has max_len >= min_len tokens)."""
    cap = [int(x) for x in cap]
    bs = set(int(x) for x in (banned or []))
    assert not any(x in bs for x in cap[prefix_len:]), (cap, bs)
    n = int(no_repeat_ngram)
    if n >= 1:
        for e in range(max(prefix_len, n - 1), len(cap)):
            g = cap[e - n + 1:e + 1]
            assert not any(cap[j:j + n] == g for j in range(0, e - n + 1)), (cap, n, e)
    assert len(cap) >= min_len, (cap, min_len)
