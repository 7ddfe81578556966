"""Caption scoring (fpnmt_score, include/fpnmt.h) on the CPU: the definition pinned on the oracle.

Scoring a sampled caption is the uncached teacher-forced pass over [<start>] + caption: its terms log_softmax(z_j)[target_j]
(targets: the caption, then <end> unless the caption ran max_len steps) must add up to the log-likelihood the KV-cached
sampler accumulated for it.  Both run in fp64 on the same weights and memory; they differ in the order of their sums and in
where they round: teacher_forced_logprobs returns fp32 log-probabilities (each term within ~1 fp32 ulp of its value), the
sampler sums fp64 log-probabilities of fp32 logits.  So the bound is a few fp32 ulps of the sum of the terms' magnitudes:
4 * 2^-23 * sum |term| (each term carries <= 1 ulp from the fp32 logits and <= 1 from the fp32 log_softmax, with margin).
"""
import numpy as np
import torch

import fpnmt_oracle as O
import sample_oracle as SO

BB, S, L, V, T, N, B = "mobilenet224_1.0", 256, 2, 512, 16, 4, 4


def test_sum_of_teacher_forced_terms_is_the_sample_logprob():
    w = O.caption_weights(BB, vocab=V, layers=L, seed=0, end_bias=6.0)
    W64 = O.W(w, torch.float64)
    img = O.test_images(B, S, seed=41)
    with torch.no_grad():
        mem = O.encoder(img, W64, BB, num_layers=L, input_vocab_size=(S // 16) ** 2)
        ids, lens, lp = SO.sample_batch_cached(mem, W64, T, N, 2, 3, temperature=1.0, top_p=0.9, seed=7, num_layers=L)
    assert ((lens > 0) & (lens < T)).sum() >= 2 and (lens == T).any()      # captions with an <end> term and truncated ones
    assert len({tuple(ids[b, n, :lens[b, n]]) for b in range(B) for n in range(N)}) > B        # the samples differ
    worst = 0.0
    for b in range(B):
        for n in range(N):
            ln = int(lens[b, n])
            cap = [int(x) for x in ids[b, n, :ln]]
            tgt = cap + ([3] if ln < T else [])
            tok = torch.tensor([[2] + cap[:len(tgt) - 1]])
            with torch.no_grad():
                tl = O.teacher_forced_logprobs(mem[b:b + 1], tok, W64, T, L)[0]
            terms = tl[torch.arange(len(tgt)), torch.tensor(tgt)].double()
            err = abs(float(terms.sum()) - float(lp[b, n]))
            bound = 4 * 2.0 ** -23 * float(terms.abs().sum())
            worst = max(worst, err / bound)
            assert err <= bound, (b, n, err, bound)
    print("worst error / bound: %.3f" % worst)
