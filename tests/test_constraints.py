"""Constrained decoding (fpnmt_beam_search_constrained / fpnmt_sample_constrained, include/fpnmt.h) on the CPU: the definition
pinned on the fp64 oracle, restated in tests/constraint_oracle.py.

Subject: that of test_prefix.py (V 512, T 12, B 8, <end> bias 12) at N = 4.
"""
import numpy as np
import pytest
import torch

import fpnmt_oracle as O
import constraint_oracle as CO
import prefix_oracle as PO
import sample_oracle as SO
import beam_search_oracle as BO

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
    # the unconstrained beams' most frequent tokens: banning them changes the search
    ids, lens, _ = BO.beam_search_nbest(mem, W64, T, N, 2, 3, num_layers=L)
    toks = np.concatenate([ids[b, n, :lens[b, n]] for b in range(B) for n in range(N)])
    banned = [int(x) for x in np.argsort(-np.bincount(toks, minlength=V), kind="stable")[:3]]
    return dict(W64=W64, mem=mem, prefix=prefix, plen=plen, banned=banned)


def _brute_ban(w, V, end, n, min_len, banned):
    """A(t) by enumeration: v is banned when it is listed, when it is <end> before min_len tokens, or when appending it makes
    the caption's last n-gram occur earlier."""
    t = len(w)
    a = np.zeros(V, bool)
    for v in range(V):
        if v in banned or (v == end and t < min_len):
            a[v] = True
        elif n >= 1 and t + 1 >= n:
            c = list(w) + [v]
            g = c[t + 1 - n:]
            a[v] = any(c[j:j + n] == g for j in range(0, t + 1 - n))
    return a


@pytest.mark.parametrize("n", [1, 2, 3, 4])
def test_ban_set_matches_enumeration(n):
    rng = np.random.default_rng(n)
    Vs = 12
    for _ in range(60):
        w = [int(x) for x in rng.integers(0, 4, size=rng.integers(0, 14))]   # four ids: many repeats
        banned = [int(x) for x in rng.choice(np.arange(4, Vs), size=2, replace=False)]
        min_len = int(rng.integers(0, 10))
        a = CO.ban_set(w, Vs, 11, n, min_len, banned)
        assert np.array_equal(a, _brute_ban(w, Vs, 11, n, min_len, banned)), (w, n, min_len)


def test_ban_set_counts_prefix_tokens():
    # a forced prefix is part of the history: the repeat of its bigram is banned, and it counts toward min_len
    assert CO.ban_set([7, 8, 9, 7], 16, 3, no_repeat_ngram=2)[8]
    assert not CO.ban_set([7, 8, 9, 7], 16, 3, no_repeat_ngram=2, min_len=4)[3]
    assert CO.ban_set([7, 8, 9], 16, 3, min_len=4)[3]


@pytest.mark.parametrize("g,lam", [(1, 0.0), (2, 0.5)])
def test_all_off_is_the_prefix_and_unprompted_search(subject, g, lam):
    s = subject
    a = CO.constrained_beam_search(s["mem"], s["W64"], T, N, g, lam, 2, 3, prefix=s["prefix"], prefix_len=s["plen"],
                                   length_penalty=0.8, num_layers=L)
    ref = PO.prefix_beam_search(s["mem"], s["W64"], T, N, g, lam, 2, 3, s["prefix"], s["plen"], length_penalty=0.8, num_layers=L)
    for x, y in zip(a, ref):
        assert np.array_equal(x, y)
    if g == 1:
        a = CO.constrained_beam_search(s["mem"], s["W64"], T, N, 1, 0.0, 2, 3, num_layers=L)
        for x, y in zip(a, BO.beam_search_nbest(s["mem"], s["W64"], T, N, 2, 3, num_layers=L)):
            assert np.array_equal(x, y)


def test_all_off_is_the_prefix_and_unprompted_sampler(subject):
    s = subject
    a = CO.constrained_sample(s["mem"], s["W64"], T, N, 2, 3, prefix=s["prefix"], prefix_len=s["plen"], num_layers=L, **SAMPLING)
    ref = PO.prefix_sample(s["mem"], s["W64"], T, N, 2, 3, s["prefix"], s["plen"], num_layers=L, **SAMPLING)
    for x, y in zip(a, ref):
        assert np.array_equal(x, y)
    a = CO.constrained_sample(s["mem"], s["W64"], T, N, 2, 3, num_layers=L, **SAMPLING)
    for x, y in zip(a, SO.sample_batch_cached(s["mem"], s["W64"], T, N, 2, 3, num_layers=L, **SAMPLING)):
        assert np.array_equal(x, y)


def _teacher_forced(s, b, cap, ln):
    tgt = list(cap) + ([3] if ln < T else [])
    tok = torch.tensor([[2] + list(cap[:len(tgt) - 1])])
    with torch.no_grad():
        tl = O.teacher_forced_logprobs(s["mem"][b:b + 1], tok, s["W64"], T, L)[0]
    terms = tl[torch.arange(len(tgt)), torch.tensor(tgt)].double()
    return float(terms.sum()), float(terms.abs().sum())


@pytest.mark.parametrize("g,lam,prompted", [(1, 0.0, False), (2, 0.5, True)])
def test_constrained_beams_obey_and_keep_their_logprob(subject, g, lam, prompted):
    s = subject
    con = dict(no_repeat_ngram=2, min_len=5, banned=s["banned"])
    pfx = dict(prefix=s["prefix"], prefix_len=s["plen"]) if prompted else {}
    ids, lens, lp = CO.constrained_beam_search(s["mem"], s["W64"], T, N, g, lam, 2, 3, length_penalty=0.8, num_layers=L,
                                               **pfx, **con)
    ref = CO.constrained_beam_search(s["mem"], s["W64"], T, N, g, lam, 2, 3, length_penalty=0.8, num_layers=L, **pfx)
    assert not np.array_equal(ids, ref[0])                   # the constraints bite on this subject
    for b in range(B):
        k = int(s["plen"][b]) if prompted else 0
        assert (ids[b, :, :k] == s["prefix"][b, :k]).all()
        for n in range(N):
            cap = ids[b, n, :lens[b, n]]
            CO.check_caption(cap, 2, 5, s["banned"], k)
            tot, mag = _teacher_forced(s, b, cap, int(lens[b, n]))
            assert abs(tot - float(lp[b, n])) <= 8 * 2.0 ** -23 * (mag + 100.0), (b, n, tot, lp[b, n])
    es = CO.constrained_beam_search(s["mem"], s["W64"], T, N, g, lam, 2, 3, length_penalty=0.8, early_stop=False,
                                    num_layers=L, **pfx, **con)
    for x, y in zip((ids, lens, lp), es):
        assert np.array_equal(x, y)


@pytest.mark.parametrize("sampling", [SAMPLING, dict(temperature=0.0), dict(temperature=0.7, top_k=5, seed=3)])
def test_constrained_samples_obey_and_keep_their_logprob(subject, sampling):
    s = subject
    con = dict(no_repeat_ngram=1, min_len=4, banned=s["banned"])
    ids, lens, lp = CO.constrained_sample(s["mem"], s["W64"], T, N, 2, 3, prefix=s["prefix"], prefix_len=s["plen"],
                                          num_layers=L, **con, **sampling)
    for b in range(B):
        k = int(s["plen"][b])
        assert (ids[b, :, :k] == s["prefix"][b, :k]).all()
        for n in range(N):
            cap = ids[b, n, :lens[b, n]]
            CO.check_caption(cap, 1, 4, s["banned"], k)
            tot, mag = _teacher_forced(s, b, cap, int(lens[b, n]))
            assert abs(tot - float(lp[b, n])) <= 4 * 2.0 ** -23 * mag, (b, n)


def test_banned_top_token_yields_the_next_allowed_with_its_unmasked_score():
    V_, end = 10, 3
    logits = np.array([[0.0, 5.0, 4.0, -1.0, 3.0, 2.0, 1.0, 0.5, 0.2, 0.1],
                       [0.0] * 10], np.float32)
    score = np.array([0.0, -np.inf], np.float32)
    fin = np.zeros(2, np.int64)
    lp = np.ones(T + 2)
    ban = np.zeros((2, V_), bool)
    ban[:, 1] = True                                            # the arg-max
    parent, token, new, _ = CO.constrained_diverse_step(logits, score, fin, lp, 0, end, 1, 0.0, ban)
    ls = torch.log_softmax(torch.from_numpy(logits[0]), -1).numpy()
    assert list(token) == [2, 4] and list(parent) == [0, 0]
    assert new[0] == np.float32(ls[2]) and new[1] == np.float32(ls[4])
    # the same step without the ban ranks token 1 first
    _, token0, _, _ = CO.constrained_diverse_step(logits, score, fin, lp, 0, end, 1, 0.0, np.zeros((2, V_), bool))
    assert list(token0) == [1, 2]


def test_greedy_and_top_k_skip_banned_maxima():
    z = np.array([1.0, 9.0, 8.0, 7.0, 2.0, 7.0], np.float32)
    ban = np.zeros(6, bool)
    ban[[1, 2]] = True
    lse = float(np.log(np.exp(z.astype(np.float64)).sum()))
    r = CO.constrained_sample_step(z, 0, 0, 0, dict(temperature=0.0), ban)
    assert r["token"] == 3 and abs(r["logprob"] - (7.0 - lse)) < 1e-12     # lowest id among the allowed maxima
    for seed in range(20):
        r = CO.constrained_sample_step(z, 0, 0, 0, dict(temperature=1.0, top_k=2, seed=seed), ban)
        assert r["token"] in (3, 5)                                        # the 2 largest ALLOWED logits (7, 7)
        assert r["K1"][[3, 5]].all() and not r["K2"][[0, 1, 2, 4]].any()
        assert abs(r["logprob"] - (float(z[r["token"]]) - lse)) < 1e-12
