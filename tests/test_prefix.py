"""Prompted decoding (fpnmt_beam_search_prefix / fpnmt_sample_prefix, include/fpnmt.h) on the CPU: the definition pinned on
the fp64 oracle, restated in tests/prefix_oracle.py.

Subject: that of test_diverse_beam_search.py (V 512, T 12, B 8, <end> bias 12) at N = 4, prefix lengths 0 .. 3 mixed across
images.  Log-likelihood bound: that of test_diverse_beam_search.py, 2^-23 * (2 * sum_j max|z_j| + n * sum_j |term_j|).
"""
import numpy as np
import pytest
import torch

import fpnmt_oracle as O
from fpnmt_oracle.model import create_look_ahead_mask, transformer_logits
import beam_search_oracle as BO
import diverse_beam_oracle as DO
import prefix_oracle as PO
import sample_oracle as SO

BB, S, L, V, T, B, N = "mobilenet224_1.0", 256, 2, 512, 12, 8, 4
SAMPLING = dict(temperature=1.0, top_k=0, top_p=0.9, seed=7)


@pytest.fixture(scope="module")
def subject():
    w = O.caption_weights(BB, vocab=V, layers=L, seed=0, end_bias=12.0)
    W64 = O.W(w, torch.float64)
    img = O.test_images(B, S, seed=41)
    with torch.no_grad():
        mem = O.encoder(img, W64, BB, num_layers=L, input_vocab_size=(S // 16) ** 2)
    rng = np.random.default_rng(5)
    prefix = rng.integers(4, V, size=(B, 3)).astype(np.int32)
    plen = (np.arange(B) % 4).astype(np.int32)
    return dict(W64=W64, mem=mem, prefix=prefix, plen=plen)


def _caps(ids, lens, b):
    return [tuple(int(x) for x in ids[b, n, :lens[b, n]]) for n in range(ids.shape[1])]


@pytest.mark.parametrize("g,lam,alpha", [(1, 0.0, 0.0), (1, 0.0, 0.8), (2, 0.5, 0.8)])
def test_empty_prefixes_are_the_unprompted_search(subject, g, lam, alpha):
    s = subject
    zero = np.zeros(B, np.int32)
    a = PO.prefix_beam_search(s["mem"], s["W64"], T, N, g, lam, 2, 3, s["prefix"], zero, length_penalty=alpha, num_layers=L)
    if g == 1:
        ref = BO.beam_search_nbest(s["mem"], s["W64"], T, N, 2, 3, length_penalty=alpha, num_layers=L)
    else:
        ref = DO.diverse_beam_search(s["mem"], s["W64"], T, N, g, lam, 2, 3, length_penalty=alpha, num_layers=L)
    for x, y in zip(a, ref):
        assert np.array_equal(x, y)


def test_empty_prefixes_are_the_unprompted_sampler(subject):
    s = subject
    a = PO.prefix_sample(s["mem"], s["W64"], T, N, 2, 3, s["prefix"], np.zeros(B, np.int32), num_layers=L, **SAMPLING)
    ref = SO.sample_batch_cached(s["mem"], s["W64"], T, N, 2, 3, num_layers=L, **SAMPLING)
    for x, y in zip(a, ref):
        assert np.array_equal(x, y)


def _teacher_forced_check(s, ids, lens, lp):
    worst = 0.0
    for b in range(B):
        for n in range(N):
            ln = int(lens[b, n])
            cap = [int(x) for x in ids[b, n, :ln]]
            tgt = cap + ([3] if ln < T else [])
            tok = torch.tensor([[2] + cap[:len(tgt) - 1]])
            with torch.no_grad():
                z, _ = transformer_logits(s["mem"][b:b + 1], tok, s["W64"], create_look_ahead_mask(len(tgt), torch.float64), T,
                                          num_layers=L)
            z = z[0].double()
            terms = torch.log_softmax(z, -1)[torch.arange(len(tgt)), torch.tensor(tgt)]
            err = abs(float(terms.sum()) - float(lp[b, n]))
            bound = 2.0 ** -23 * (2 * float(z.abs().max(-1).values.sum()) + len(tgt) * float(terms.abs().sum()))
            worst = max(worst, err / bound)
            assert err <= bound, (b, n, err, bound)
    print("worst error / bound: %.3f" % worst)


@pytest.mark.parametrize("g,lam", [(1, 0.0), (2, 0.5)])
def test_beams_carry_the_prefix_and_their_logprob(subject, g, lam):
    s = subject
    ids, lens, lp = PO.prefix_beam_search(s["mem"], s["W64"], T, N, g, lam, 2, 3, s["prefix"], s["plen"], length_penalty=0.8,
                                          num_layers=L)
    m = N // g
    for b in range(B):
        k = int(s["plen"][b])
        assert (lens[b] >= k).all()
        assert (ids[b, :, :k] == s["prefix"][b, :k]).all()
        for q in range(g):
            caps = _caps(ids, lens, b)[q * m:(q + 1) * m]
            assert len(set(caps)) == m
    assert not (ids * (np.arange(T)[None, None, :] >= lens[..., None])).any()
    _teacher_forced_check(s, ids, lens, lp)
    es = PO.prefix_beam_search(s["mem"], s["W64"], T, N, g, lam, 2, 3, s["prefix"], s["plen"], length_penalty=0.8,
                               early_stop=False, num_layers=L)
    for x, y in zip((ids, lens, lp), es):
        assert np.array_equal(x, y)


def test_samples_carry_the_prefix_and_their_logprob(subject):
    s = subject
    ids, lens, lp = PO.prefix_sample(s["mem"], s["W64"], T, N, 2, 3, s["prefix"], s["plen"], num_layers=L, **SAMPLING)
    for b in range(B):
        k = int(s["plen"][b])
        assert (lens[b] >= k).all() and (ids[b, :, :k] == s["prefix"][b, :k]).all()
    # the fp64 sampler sums fp64 terms of fp32 logits: the bound of test_scoring.py
    for b in range(B):
        for n in range(N):
            ln = int(lens[b, n])
            cap = [int(x) for x in ids[b, n, :ln]]
            tgt = cap + ([3] if ln < T else [])
            tok = torch.tensor([[2] + cap[:len(tgt) - 1]])
            with torch.no_grad():
                tl = O.teacher_forced_logprobs(s["mem"][b:b + 1], tok, s["W64"], T, L)[0]
            terms = tl[torch.arange(len(tgt)), torch.tensor(tgt)].double()
            assert abs(float(terms.sum()) - float(lp[b, n])) <= 4 * 2.0 ** -23 * float(terms.abs().sum()), (b, n)


@pytest.mark.parametrize("k", [1, 3])
def test_own_prefix_reproduces_sample_zero(subject, k):
    s = subject
    ref = SO.sample_batch_cached(s["mem"], s["W64"], T, N, 2, 3, num_layers=L, **SAMPLING)
    ids0, lens0, lp0 = ref
    ok = lens0[:, 0] >= k
    assert ok.sum() >= B // 2
    prefix = np.zeros((B, k), np.int32)
    prefix[ok] = ids0[ok, 0, :k]
    plen = np.where(ok, k, 0).astype(np.int32)
    ids, lens, lp = PO.prefix_sample(s["mem"], s["W64"], T, N, 2, 3, prefix, plen, num_layers=L, **SAMPLING)
    assert np.array_equal(ids[:, 0], ids0[:, 0]) and np.array_equal(lens[:, 0], lens0[:, 0])
    assert np.array_equal(lp[:, 0], lp0[:, 0])
    assert np.array_equal(ids[~ok], ids0[~ok])                      # images without a prefix are untouched
