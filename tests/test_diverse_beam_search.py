"""Diverse beam search (fpnmt_beam_search_diverse, include/fpnmt.h) on the CPU: the definition pinned on the fp64 oracle,
restated in tests/diverse_beam_oracle.py.

Subject: that of test_beam_search.py (V 512, T 12, B 8, <end> bias 12), at N = 4 with G = 2 and 4 and at N = 8 with G = 4.
The restatement ranks every candidate of a row; the engine ranks only each row's N best (the penalty only lowers keys and at
most N - N / G tokens carry one, see DESIGN.md), so where the two agree here the sufficiency argument is what the GPU tests
then lean on.  Log-likelihood bound: that of test_beam_search.py, 2^-23 * (2 * sum_j max|z_j| + n * sum_j |term_j|).
"""
import numpy as np
import pytest
import torch

import fpnmt_oracle as O
from fpnmt_oracle.model import create_look_ahead_mask, transformer_logits
import beam_search_oracle as BO
import diverse_beam_oracle as DO

BB, S, L, V, T, B = "mobilenet224_1.0", 256, 2, 512, 12, 8
CASES = [(4, 2), (4, 4), (8, 4)]          # (N, G)


@pytest.fixture(scope="module")
def subject():
    w = O.caption_weights(BB, vocab=V, layers=L, seed=0, end_bias=12.0)
    W64 = O.W(w, torch.float64)
    img = O.test_images(B, S, seed=41)
    with torch.no_grad():
        mem = O.encoder(img, W64, BB, num_layers=L, input_vocab_size=(S // 16) ** 2)
    runs = {}

    def run(n, g, lam, alpha=0.0, es=True, t=T):
        k = (n, g, lam, alpha, es, t)
        if k not in runs:
            runs[k] = DO.diverse_beam_search(mem, W64, t, n, g, lam, 2, 3, length_penalty=alpha, early_stop=es, num_layers=L)
        return runs[k]
    return dict(W64=W64, mem=mem, run=run)


def _caps(ids, lens, b, rng):
    return [tuple(ids[b, n, :lens[b, n]]) for n in rng]


@pytest.mark.parametrize("alpha", [0.0, 0.8])
@pytest.mark.parametrize("lam", [0.0, 0.5, 1e4])
def test_one_group_is_the_nbest_search(subject, lam, alpha):
    a = subject["run"](4, 1, lam, alpha)
    ref = BO.beam_search_nbest(subject["mem"], subject["W64"], T, 4, 2, 3, length_penalty=alpha, num_layers=L)
    for x, y in zip(a, ref):
        assert np.array_equal(x, y)


@pytest.mark.parametrize("n,g", CASES)
def test_zero_diversity_repeats_the_narrow_search_in_every_group(subject, n, g):
    ids, lens, lp = subject["run"](n, g, 0.0)
    m = n // g
    ref = BO.beam_search_nbest(subject["mem"], subject["W64"], T, m, 2, 3, num_layers=L)
    for k in range(g):
        for x, y in zip((ids, lens, lp), ref):
            assert np.array_equal(x[:, k * m:(k + 1) * m], y)


@pytest.mark.parametrize("n,g", CASES)
def test_huge_diversity_at_one_step_gives_the_top_tokens_in_group_major_order(subject, n, g):
    """max_len = 1: each caption is its step-0 token (empty for <end>).  With lambda far above any log-prob gap, group g can
    only take tokens no earlier group took, so the N captions are the N most likely first tokens in order."""
    ids, lens, lp = subject["run"](n, g, 1e4, 0.0, True, 1)
    with torch.no_grad():
        tf = O.teacher_forced_logprobs(subject["mem"], torch.full((B, 1), 2, dtype=torch.int64), subject["W64"], T,
                                       L)[:, 0].double().numpy()
    checked = 0
    for b in range(B):
        top = np.argsort(-tf[b], kind="stable")[:n + 1]
        if np.diff(tf[b, top]).max() > -1e-5:                         # near tie: fp32 against fp64 may order it differently
            continue
        checked += 1
        for k in range(n):
            tok = int(top[k])
            assert lens[b, k] == (0 if tok == 3 else 1), (b, k)
            assert tok == 3 or ids[b, k, 0] == tok, (b, k)
            assert abs(float(lp[b, k]) - tf[b, tok]) <= 1e-5 * max(1.0, abs(tf[b, tok])), (b, k)
    assert checked >= B - 1


@pytest.mark.parametrize("n,g", [(4, 2), (4, 4)])
def test_diversity_gives_more_distinct_captions(subject, n, g):
    def distinct(r):
        return sum(len(set(_caps(r[0], r[1], b, range(n)))) for b in range(B))
    d0, d5 = distinct(subject["run"](n, g, 0.0)), distinct(subject["run"](n, g, 0.5))
    print("N=%d G=%d: %d distinct captions at lambda 0, %d at 0.5 (of %d)" % (n, g, d0, d5, B * n))
    assert d5 > d0


@pytest.mark.parametrize("alpha", [0.0, 0.8])
@pytest.mark.parametrize("n,g", CASES)
def test_structure(subject, n, g, alpha):
    ids, lens, lp = subject["run"](n, g, 0.5, alpha)
    m = n // g
    table = BO.length_penalty_table(T, alpha)
    assert (lens < T).any() and (lens == T).any()
    for b in range(B):
        key = [np.float32(lp[b, k]) / table[min(int(lens[b, k]) + 1, T)] for k in range(n)]
        for k in range(g):
            grp = range(k * m, (k + 1) * m)
            assert all(key[i] >= key[i + 1] for i in grp[:-1]), (b, key)
            caps = _caps(ids, lens, b, grp)
            assert len(set(caps)) == m
            assert all(3 not in c for c in caps)
        assert ((lens[b] >= 0) & (lens[b] <= T)).all()
        assert not (ids[b] * (np.arange(T)[None, :] >= lens[b][:, None])).any()


@pytest.mark.parametrize("n,g", CASES)
def test_logprob_is_the_teacher_forced_sum(subject, n, g):
    ids, lens, lp = subject["run"](n, g, 0.5, 0.8)
    worst = 0.0
    for b in range(B):
        for k in range(n):
            ln = int(lens[b, k])
            cap = [int(x) for x in ids[b, k, :ln]]
            tgt = cap + ([3] if ln < T else [])
            tok = torch.tensor([[2] + cap[:len(tgt) - 1]])
            with torch.no_grad():
                z, _ = transformer_logits(subject["mem"][b:b + 1], tok, subject["W64"],
                                          create_look_ahead_mask(len(tgt), torch.float64), T, num_layers=L)
            z = z[0].double()
            terms = torch.log_softmax(z, -1)[torch.arange(len(tgt)), torch.tensor(tgt)]
            err = abs(float(terms.sum()) - float(lp[b, k]))
            bound = 2.0 ** -23 * (2 * float(z.abs().max(-1).values.sum()) + len(tgt) * float(terms.abs().sum()))
            worst = max(worst, err / bound)
            assert err <= bound, (b, k, err, bound)
    print("worst error / bound: %.3f" % worst)


@pytest.mark.parametrize("n,g", CASES)
def test_early_stop_equals_the_full_run(subject, n, g):
    a, b = subject["run"](n, g, 0.5, 0.8, True), subject["run"](n, g, 0.5, 0.8, False)
    assert (a[1] < T).all(1).any()                                   # an image closes before the last step
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
