"""Sampled caption decoding (fpnmt_sampling, include/fpnmt.h) on the CPU: the fp64 oracle of tests/sample_oracle.py against
hand-built logits, Philox known answers, the ctypes mirror of the parameter struct, and the oracle's greedy decode against its
beam search."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

import fpnmt_oracle as O
import sample_oracle as SO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _hex(words):
    return " ".join("%08x" % int(x) for x in words)


def test_philox_known_answers():
    assert _hex(SO.philox4x32_10([0, 0, 0, 0], [0, 0])) == "6627e8d5 e169c58d bc57ac4c 9b00dbd8"
    ones = 0xFFFFFFFF
    assert _hex(SO.philox4x32_10([ones] * 4, [ones] * 2)) == "408f276d 41c83b0e a20bc7c6 6d5451fd"
    assert _hex(SO.philox4x32_10([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0])) == \
        "d16cfe09 94fdcceb 5001e420 24126ea1"
    # batched form == one call per counter; u is a multiple of 2^-24 in [0, 1)
    ctr = np.array([[t, 3, 5, 0] for t in range(7)], np.uint64)
    many = SO.philox4x32_10(ctr, np.array([[11, 0]] * 7, np.uint64))
    for i in range(7):
        assert (many[i] == SO.philox4x32_10(ctr[i], [11, 0])).all()
    u = SO.uniform(2, 1, 0, 12345)
    assert 0.0 <= u < 1.0 and (u * 2 ** 24) == int(u * 2 ** 24)


def _p(**kw):
    d = dict(temperature=1.0, top_k=0, top_p=1.0, seed=0)
    d.update(kw)
    return d


def test_ties_at_the_kth_logit_are_all_kept():
    z = np.array([5.0, 4.0, 3.0, 3.0, 3.0, 1.0, 0.5, 0.0])
    r = SO.sample_step(z, 0, 0, 0, _p(top_k=3))
    assert r["K1"].tolist() == [True] * 5 + [False] * 3            # |K1| = 5 > k: the three tokens at z_(3) stay
    assert r["K2"].tolist() == r["K1"].tolist()
    r = SO.sample_step(z, 0, 0, 0, _p(top_k=2))
    assert r["K1"].tolist() == [True, True] + [False] * 6


def test_ties_at_the_nucleus_boundary_are_all_kept():
    z = np.log(np.array([0.4, 0.2, 0.2, 0.1, 0.1]))
    # 0.4 alone < 0.5; 0.4 + one 0.2 >= 0.5: tau = 0.2 and both tokens at 0.2 stay
    r = SO.sample_step(z, 0, 0, 0, _p(top_p=0.5))
    assert r["K2"].tolist() == [True, True, True, False, False]
    np.testing.assert_allclose(r["q"], [0.5, 0.25, 0.25, 0, 0], atol=1e-12)          # renormalised over K2
    r = SO.sample_step(z, 0, 0, 0, _p(top_p=0.85))
    assert r["K2"].tolist() == [True] * 5                                             # the two 0.1 tie at the cut


def test_top_p_to_zero_keeps_only_the_argmax_set():
    z = np.array([1.0, 3.0, 2.0, 3.0, -1.0])
    for t in range(20):
        r = SO.sample_step(z, 0, 0, t, _p(top_p=1e-9, temperature=1.3, seed=t))
        assert r["K2"].tolist() == [False, True, False, True, False]
        assert r["token"] in (1, 3)


def test_top_k_v_with_top_p_one_is_plain_sampling():
    rng = np.random.default_rng(0)
    z = rng.normal(size=40)
    for temp in (0.5, 1.0, 1.7):
        r = SO.sample_step(z, 2, 1, 4, _p(top_k=40, temperature=temp, seed=9))
        q = np.exp(z / temp - (z / temp).max())
        q /= q.sum()
        assert r["K2"].all()
        np.testing.assert_allclose(r["q"], q, rtol=1e-12)
        c = np.cumsum(q)
        assert r["token"] == int(np.argmax(c > r["u"]))                              # the first CDF step above u


def test_padded_entries_are_never_drawn():
    rng = np.random.default_rng(1)
    z = rng.normal(size=64)
    z[50:] = -1e9                                                                     # Pipeline's padded vocabulary
    for t in range(300):
        for params in (_p(seed=t), _p(top_k=64, seed=t), _p(temperature=5.0, seed=t), _p(top_p=0.999999, seed=t)):
            r = SO.sample_step(z, t % 3, t % 5, t, params)
            assert r["token"] < 50 and (r["q"][50:] == 0).all()


def test_temperature_changes_k2_but_not_k1():
    z = np.array([3.0, 2.5, 2.0, 1.5, 1.0, 0.5, 0.0, -0.5])
    cold = SO.sample_step(z, 0, 0, 0, _p(top_k=5, top_p=0.6, temperature=0.5))
    hot = SO.sample_step(z, 0, 0, 0, _p(top_k=5, top_p=0.6, temperature=2.0))
    assert cold["K1"].tolist() == hot["K1"].tolist() == [True] * 5 + [False] * 3
    assert cold["K2"].sum() < hot["K2"].sum()                                         # a hotter nucleus is wider
    # the log-probability is taken at temperature 1 without filtering, whatever the sampling parameters
    for r in (cold, hot):
        assert abs(r["logprob"] - (z[r["token"]] - np.log(np.exp(z).sum()))) < 1e-12


def test_draw_on_an_exact_cdf_step_takes_the_next_token():
    # u = 1/2, 3/4, 1/4 exactly (seeds found by search): four equal logits, cumulative mass u * 4 reached at token 4u - 1,
    # exceeded first at token 4u
    z = np.array([0.0] * 4 + [-1e9] * 4)
    for seed, uu in [(515707, 0.5), (22356995, 0.75), (23739184, 0.25)]:
        r = SO.sample_step(z, 0, 0, 0, _p(seed=seed))
        assert r["u"] == uu and r["token"] == int(4 * uu)


def test_greedy_is_the_lowest_argmax():
    z = np.array([0.0, 2.0, 1.0, 2.0])
    for t in range(5):
        assert SO.sample_step(z, 0, t, t, _p(temperature=0.0, seed=t))["token"] == 1


def test_sampling_struct_mirror_matches_the_header(tmp_path):
    from fpnmt import _lib
    src = tmp_path / "probe.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "fpnmt.h"\nint main(void) {\n'
                   '  printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(fpnmt_sampling), offsetof(fpnmt_sampling, temperature),\n'
                   '         offsetof(fpnmt_sampling, top_k), offsetof(fpnmt_sampling, top_p), offsetof(fpnmt_sampling, seed),\n'
                   '         offsetof(fpnmt_sampling, reserved));\n  return 0;\n}\n')
    exe = tmp_path / "probe"
    r = subprocess.run(["gcc", "-std=c11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True).stdout.split()]
    S = _lib.FpnmtSampling
    assert got == [C.sizeof(S), S.temperature.offset, S.top_k.offset, S.top_p.offset, S.seed.offset, S.reserved.offset]
    sp = _lib.sampling(0.7, 10, 0.9, -1)
    assert sp.seed == 0xFFFFFFFFFFFFFFFF and list(sp.reserved) == [0] * 4


BB, S, L, V, T, N, B = "mobilenet224_1.0", 256, 2, 512, 12, 3, 4


@pytest.fixture(scope="module")
def subject():
    w = O.caption_weights(BB, vocab=V, layers=L, seed=0, end_bias=6.0)
    Wv = O.W(w)
    img = O.test_images(B, S, seed=41)
    with torch.no_grad():
        mem = O.encoder(img, Wv, BB, num_layers=L, input_vocab_size=(S // 16) ** 2)
    return dict(w=w, Wv=Wv, mem=mem)


def test_oracle_greedy_equals_the_reference_beam_search(subject):
    s = subject
    ids, lens, lp = SO.sample_batch_cached(s["mem"], s["Wv"], T, N, 2, 3, temperature=0.0, seed=5, num_layers=L)
    ref_ids, ref_len = O.predict_batch_cached(s["mem"], s["Wv"], T, N, 2, 3, num_layers=L)
    for n in range(N):
        assert (ids[:, n] == ref_ids).all() and (lens[:, n] == ref_len).all()
    assert (lens < T).any() and (lens > 1).any()                                     # <end> fires, captions are not empty
    assert (lp < 0).all()


def test_oracle_samples_are_independent_rows(subject):
    """Sample n of image b depends on (seed, t, b, n) only: the same rows come out of a batch with the images reordered."""
    s = subject
    kw = dict(temperature=1.0, top_k=0, top_p=0.9, seed=3, num_layers=L)
    ids, lens, lp = SO.sample_batch_cached(s["mem"], s["Wv"], T, N, 2, 3, **kw)
    assert len({tuple(ids[b, n, :lens[b, n]]) for b in range(B) for n in range(N)}) > B     # the N samples differ
    one, one_len, one_lp = SO.sample_batch_cached(s["mem"][:1], s["Wv"], T, N, 2, 3, **kw)
    assert (one[0] == ids[0]).all() and (one_len[0] == lens[0]).all()
    np.testing.assert_allclose(one_lp[0], lp[0], rtol=1e-6)
