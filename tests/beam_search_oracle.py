"""N-best beam search (fpnmt_beam_search, include/fpnmt.h) restated on the oracle.  TEST INFRASTRUCTURE ONLY.

`beam_search_nbest` does not decode on its own: it runs `fpnmt_oracle.decode.predict_batch_cached` with the true-beam start
and frozen finished beams over all max_seq_len steps, records the logits of every step, and replays the search with the
same `_beam_step_finished` on them.  The replay therefore follows exactly the beams the cached decode followed; what it adds
is the N-best close: an image is finished when all N of its beams are frozen (early_stop=True) or after max_seq_len steps,
and then every beam is read out in slot order, which is rank order.
"""
from __future__ import annotations

from typing import Tuple

import numpy as np
import torch

from fpnmt_oracle.decode import _beam_step_finished, predict_batch_cached


def length_penalty_table(max_seq_len: int, alpha: float) -> np.ndarray:
    """lp[n] = ((5 + n) / 6) ** alpha for n = 0 .. max_seq_len + 1, as predict_batch_cached computes it."""
    return np.array([np.power(np.float32((5.0 + i) / 6.0), np.float32(alpha)) for i in range(max_seq_len + 2)], np.float32)


def beam_search_nbest(enc_output: torch.Tensor, w, max_seq_len: int, beam: int, start: int, end: int,
                      length_penalty: float = 0.0, early_stop: bool = True, num_layers: int = 6,
                      num_heads: int = 8) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Returns ids (B, N, T) int32 (no <start>, no <end>, 0 from len on), lens (B, N) int32 (T: truncated) and the raw beam
    scores (B, N) float32 (sum of log_softmax terms over min(len + 1, T) positions).  early_stop=False closes every image at
    the last step instead of at the step where its last beam froze (the result must be the same)."""
    T, N = max_seq_len, beam
    trace = {}
    with torch.no_grad():
        predict_batch_cached(enc_output, w, T, N, start, end, num_layers=num_layers, num_heads=num_heads, early_stop=False,
                             trace=trace, true_beam=True, finished_beams=True, length_penalty=length_penalty)
    lp = length_penalty_table(T, length_penalty)
    bsz = enc_output.shape[0]
    ids = np.zeros((bsz, N, T), np.int32)
    lens = np.zeros((bsz, N), np.int32)
    logprob = np.zeros((bsz, N), np.float32)
    for b in range(bsz):
        seqs = np.full((N, 1), start, np.int64)
        score = np.zeros((N,), np.float32)
        score[1:] = -np.inf
        fin = np.zeros((N,), np.int64)
        for t in range(T):
            parent, token, score, fin = _beam_step_finished(trace["logits"][t][b], score, fin, lp, t, end)
            seqs = np.concatenate([seqs[parent], token[:, None]], axis=-1)
            if (early_stop and (fin > 0).all()) or t == T - 1:
                for n in range(N):
                    ln = int(fin[n]) - 1 if fin[n] > 0 else t + 1
                    ids[b, n, :ln] = seqs[n, 1:1 + ln]
                    lens[b, n] = ln
                    logprob[b, n] = score[n]
                break
    return ids, lens, logprob
