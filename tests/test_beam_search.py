"""N-best beam search (fpnmt_beam_search, include/fpnmt.h) on the CPU: the definition pinned on the fp64 oracle.

The weights stop about half of the beams before max_len, so lists hold both captions that ended with <end> (len < T) and
truncated ones (len == T), and some images finish with all their beams frozen before the last step.  A caption's
log-likelihood is checked against the uncached teacher-forced pass over [<start>] + caption.  The search sums fp32 log_softmax terms of fp32 logits in fp32, one rounding per step; each term carries
<= 1 fp32 ulp of the row's largest |logit| from the logits and about as much from the log_softmax.  So the bound is
2^-23 * (2 * sum_j max|z_j| + n * sum_j |term_j|) over the n scored positions.
"""
import numpy as np
import pytest
import torch

import fpnmt_oracle as O
from fpnmt_oracle.model import create_look_ahead_mask, transformer_logits
import beam_search_oracle as BO

BB, S, L, V, T, N, B = "mobilenet224_1.0", 256, 2, 512, 12, 4, 8


@pytest.fixture(scope="module")
def subject():
    w = O.caption_weights(BB, vocab=V, layers=L, seed=0, end_bias=12.0)
    W64 = O.W(w, torch.float64)
    img = O.test_images(B, S, seed=41)
    with torch.no_grad():
        mem = O.encoder(img, W64, BB, num_layers=L, input_vocab_size=(S // 16) ** 2)
    runs = {}
    for alpha in (0.0, 0.8):
        for es in (True, False):
            runs[alpha, es] = BO.beam_search_nbest(mem, W64, T, N, 2, 3, length_penalty=alpha, early_stop=es, num_layers=L)
    return dict(W64=W64, mem=mem, runs=runs)


def test_lists_hold_finished_and_truncated_captions(subject):
    for (alpha, _), (ids, lens, lp) in subject["runs"].items():
        assert (lens < T).any() and (lens == T).any(), (alpha, lens)
        assert (lens < T).all(axis=1).any(), (alpha, lens)          # an image closes before the last step


@pytest.mark.parametrize("alpha", [0.0, 0.8])
def test_early_stop_equals_the_full_run(subject, alpha):
    a, b = subject["runs"][alpha, True], subject["runs"][alpha, False]
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


def test_row0_is_the_finished_beams_decode(subject):
    ids, lens, _ = subject["runs"][0.0, True]
    ref_ids, ref_len = O.predict_batch_cached(subject["mem"], subject["W64"], T, N, 2, 3, num_layers=L, true_beam=True,
                                              finished_beams=True)
    assert np.array_equal(ids[:, 0], ref_ids) and np.array_equal(lens[:, 0], ref_len)


@pytest.mark.parametrize("alpha", [0.0, 0.8])
def test_structure_rank_order_and_distinct_captions(subject, alpha):
    ids, lens, lp = subject["runs"][alpha, True]
    table = BO.length_penalty_table(T, alpha)
    for b in range(B):
        key = [np.float32(lp[b, n]) / table[min(int(lens[b, n]) + 1, T)] for n in range(N)]
        assert all(key[n] >= key[n + 1] for n in range(N - 1)), (b, key)
        caps = [tuple(ids[b, n, :lens[b, n]]) for n in range(N)]
        assert len(set(caps)) == N
        for n in range(N):
            assert 0 <= lens[b, n] <= T
            assert 3 not in caps[n]
            assert not ids[b, n, lens[b, n]:].any()


@pytest.mark.parametrize("alpha", [0.0, 0.8])
def test_logprob_is_the_teacher_forced_sum(subject, alpha):
    ids, lens, lp = subject["runs"][alpha, True]
    worst = 0.0
    for b in range(B):
        for n in range(N):
            ln = int(lens[b, n])
            cap = [int(x) for x in ids[b, n, :ln]]
            tgt = cap + ([3] if ln < T else [])
            tok = torch.tensor([[2] + cap[:len(tgt) - 1]])
            with torch.no_grad():
                z, _ = transformer_logits(subject["mem"][b:b + 1], tok, subject["W64"], create_look_ahead_mask(len(tgt), torch.float64),
                                          T, num_layers=L)
            z = z[0].double()
            terms = torch.log_softmax(z, -1)[torch.arange(len(tgt)), torch.tensor(tgt)]
            err = abs(float(terms.sum()) - float(lp[b, n]))
            bound = 2.0 ** -23 * (2 * float(z.abs().max(-1).values.sum()) + len(tgt) * float(terms.abs().sum()))
            worst = max(worst, err / bound)
            assert err <= bound, (alpha, b, n, err, bound)
    print("worst error / bound: %.3f" % worst)


def test_length_penalty_changes_the_lists(subject):
    a_ids, a_len, _ = subject["runs"][0.0, True]
    b_ids, b_len, _ = subject["runs"][0.8, True]
    differ = (a_ids != b_ids).any(axis=(1, 2)) | (a_len != b_len).any(axis=1)
    assert differ.any()
