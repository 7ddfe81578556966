"""Diverse beam search (Engine.beam_search(beam_groups=G, diversity=lambda) / fpnmt_beam_search_diverse,
Pipeline.beam_search_batch) against the oracle (tests/diverse_beam_oracle.py), against `score` and against itself.

Subject: that of test_gpu_beam_search.py (S = 256, L = 2, V = 1000, T = 16, N = 8, B = 24, <end> bias 12), with G = 2, 4, 8
and lambda = 0, 0.5.

Bounds (absolute, per scored position n = min(len + 1, T)), those of test_gpu_beam_search.py:
  bf16x3  2e-3 against the oracle on the images whose whole list matches it (>= 90 % must: a list is N fragile rankings, and
          here every group's ranking also depends on the tokens the earlier groups chose), and between `score` and logprob.
  bf16    0.25 against the fp64 teacher-forced sum of the returned caption, and between `score` and logprob.
Exact (bit-equal): G = 1 against fpnmt_beam_search whatever lambda; at lambda = 0 every group of an image against every other
(rows with the same token history compute bit-identical K/V and logits, which the shared-cache design already relies on);
graphs on / off, ancestry / physical cache, default / no_kv_share, early stop on / off, two runs and engines created with
other true_beam / finished_beams / length_penalty settings; generate / sample / score / beam_search and generate's launch
count after diverse searches.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import fpnmt_oracle as O
import beam_search_oracle as BO
import diverse_beam_oracle as DO

pytestmark = pytest.mark.gpu

BB, S, L, V, T, N, B = "mobilenet224_1.0", 256, 2, 1000, 16, 8, 24
END_BIAS = 12.0
GROUPS = [2, 4, 8]


@pytest.fixture(scope="module")
def subject():
    w = O.caption_weights(BB, vocab=V, layers=L, seed=0, end_bias=END_BIAS)
    Wv = O.W(w)
    img = O.test_images(B, S, seed=41)
    with torch.no_grad():
        mem = O.encoder(img, Wv, BB, num_layers=L, input_vocab_size=(S // 16) ** 2)
    return dict(w=w, Wv=Wv, W64=O.W(w, torch.float64), img=img, mem=mem)


def _engine(s, prec="bf16", max_len=T, **kw):
    from fpnmt.engine import Engine
    return Engine(s["w"], backbone=BB, batch=B, beam=N, vocab=V, max_len=max_len, num_layers=L, image_size=S, precision=prec,
                  **kw)


def _load_memory(eng, s):
    eng.decode_logits(s["mem"].cuda(), torch.full((B, 1), 2, dtype=torch.int32).cuda())


def _search(eng, images=None, **kw):
    return [x.clone().numpy() for x in eng.beam_search(images, return_logprobs=True, **kw)]


def _n(lens):
    return np.minimum(lens + 1, T)


def _check_structure(ids, lens, lp, alpha, g):
    m = N // g
    table = BO.length_penalty_table(T, alpha)
    assert ((lens >= 0) & (lens <= T)).all()
    key = (lp.astype(np.float64) / table[_n(lens)]).reshape(B, g, m)
    # within-group rank order; the engine's table comes from powf, this one from numpy: 1 ulp of slack
    assert (key[..., :-1] >= key[..., 1:] - 2.0 ** -22 * np.abs(key[..., 1:])).all()
    for b in range(B):
        for k in range(g):
            caps = [tuple(ids[b, n, :lens[b, n]]) for n in range(k * m, (k + 1) * m)]
            assert len(set(caps)) == m, (b, k)
            assert all(3 not in c for c in caps), (b, k)
    assert not (ids * (np.arange(T)[None, None, :] >= lens[..., None])).any()   # zero past len
    assert (lp <= 0).all()


def _teacher_forced_sum(s, ids, lens):
    """fp64 sum of log_softmax terms over the n = min(len + 1, T) positions of every returned caption, (B, N)."""
    tok = np.full((B, N, T), 2, np.int64)
    tok[:, :, 1:] = ids[:, :, :T - 1]
    tgt = ids.astype(np.int64).copy()
    mask = np.arange(T)[None, None, :] < _n(lens)[..., None]
    for b in range(B):
        for n in range(N):
            if lens[b, n] < T:
                tgt[b, n, lens[b, n]] = 3
    mem = s["mem"].double().repeat_interleave(N, 0)
    with torch.no_grad():
        lp = O.teacher_forced_logprobs(mem, torch.from_numpy(tok.reshape(-1, T)), s["W64"], T, L).double().numpy()
    terms = np.take_along_axis(lp.reshape(B, N, T, -1), tgt[..., None], -1)[..., 0] * mask
    return terms.sum(-1)


def _score(eng, ids, lens):
    return eng.score(torch.from_numpy(ids).cuda(), torch.from_numpy(lens).cuda()).numpy().astype(np.float64)


def _groups_identical(out, g):
    m = N // g
    return all(np.array_equal(x.reshape(B, g, m, *x.shape[2:])[:, k], x.reshape(B, g, m, *x.shape[2:])[:, 0])
               for x in out for k in range(g))


def _diverse_raw(eng, g, lam, alpha):
    """fpnmt_beam_search_diverse called directly (Engine.beam_search takes fpnmt_beam_search for G = 1)."""
    ids = torch.zeros((B, N, T), dtype=torch.int32, device="cuda")
    lens = torch.zeros((B, N), dtype=torch.int32, device="cuda")
    lp = torch.zeros((B, N), dtype=torch.float32, device="cuda")
    rc = eng.lib.fpnmt_beam_search_diverse(eng._h, None, 0, g, C.c_float(lam), C.c_float(alpha), ids.data_ptr(),
                                           lens.data_ptr(), lp.data_ptr(), 0, 1, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return rc, [x.cpu().numpy() for x in (ids, lens, lp)]


def test_one_group_is_beam_search(subject):
    s = subject
    eng = _engine(s)
    _load_memory(eng, s)
    for alpha in (0.0, 0.8):
        ref = _search(eng, length_penalty=alpha)
        for lam in (0.0, 0.5, 7.0):
            for x, y in zip(_search(eng, length_penalty=alpha, beam_groups=1, diversity=lam), ref):
                assert np.array_equal(x, y)
            rc, out = _diverse_raw(eng, 1, lam, alpha)
            assert rc == 0
            for x, y in zip(out, ref):
                assert np.array_equal(x, y)
    eng.close()


def test_bf16x3_matches_oracle_and_score(subject):
    s = subject
    eng = _engine(s, "bf16x3")
    _load_memory(eng, s)
    for g in GROUPS:
        for lam in (0.0, 0.5):
            alpha = 0.8 if g == 4 else 0.0
            ref_ids, ref_len, ref_lp = DO.diverse_beam_search(s["mem"], s["Wv"], T, N, g, lam, 2, 3, length_penalty=alpha,
                                                              num_layers=L)
            ids, lens, lp = _search(eng, length_penalty=alpha, beam_groups=g, diversity=lam)
            sc = _score(eng, ids, lens)
            _check_structure(ids, lens, lp, alpha, g)
            same = (ids == ref_ids).all(axis=(1, 2)) & (lens == ref_len).all(axis=1)
            err = (np.abs(lp - ref_lp) / _n(lens))[same]
            print("bf16x3 G=%d lambda=%g alpha=%g: %d / %d lists identical to the oracle, worst |dlogprob| / n %.2e, "
                  "worst |score - logprob| / n %.2e" % (g, lam, alpha, same.sum(), B, err.max(),
                                                        (np.abs(sc - lp) / _n(lens)).max()))
            assert same.mean() >= 0.9, (g, lam)
            assert err.max() <= 2e-3, (g, lam)
            assert (np.abs(sc - lp) <= 2e-3 * _n(lens)).all(), (g, lam)
    eng.close()


@pytest.mark.parametrize("opts", [(), ("tgemm_wide",)])
def test_bf16_structure_likelihood_score_and_identical_groups(subject, opts):
    s = subject
    eng = _engine(s, opts=opts)
    _load_memory(eng, s)
    for g in GROUPS:
        alpha = 0.8 if g == 4 else 0.0
        zero = _search(eng, length_penalty=alpha, beam_groups=g, diversity=0.0)
        assert _groups_identical(zero, g), g
        ids, lens, lp = _search(eng, length_penalty=alpha, beam_groups=g, diversity=0.5)
        sc = _score(eng, ids, lens)
        _check_structure(ids, lens, lp, alpha, g)
        assert (lens < T).any() and (lens == T).any()
        ref = _teacher_forced_sum(s, ids, lens)
        e_ref = np.abs(lp - ref) / _n(lens)
        e_sc = np.abs(sc - lp) / _n(lens)
        distinct = [sum(len(set(tuple(x[b, n, :y[b, n]]) for n in range(N))) for b in range(B)) for x, y in
                    ((zero[0], zero[1]), (ids, lens))]
        print("bf16 %s G=%d: worst |logprob - fp64| / n %.3f, worst |score - logprob| / n %.3f; distinct captions "
              "%d at lambda 0, %d at 0.5 (of %d)" % (opts, g, e_ref.max(), e_sc.max(), distinct[0], distinct[1], B * N))
        assert e_ref.max() <= 0.25 and e_sc.max() <= 0.25
        assert distinct[1] > distinct[0]
    eng.close()


def test_huge_diversity_at_one_step_gives_the_top_tokens(subject):
    """max_len = 1, lambda = 1e4: the N captions of an image are its N most likely first tokens (empty for <end>) in
    group-major order, checked where the top N + 1 log-probs are more than 1e-3 apart."""
    s = subject
    with torch.no_grad():
        tf = O.teacher_forced_logprobs(s["mem"], torch.full((B, 1), 2, dtype=torch.int64), s["Wv"], T, L)[:, 0].double().numpy()
    eng = _engine(s, "bf16x3", max_len=1)
    _load_memory(eng, s)
    for g in GROUPS:
        ids, lens, lp = [x.clone().numpy() for x in eng.beam_search(None, beam_groups=g, diversity=1e4, return_logprobs=True)]
        checked = 0
        for b in range(B):
            top = np.argsort(-tf[b], kind="stable")[:N + 1]
            if np.diff(tf[b, top]).max() > -1e-3:
                continue
            checked += 1
            for n in range(N):
                tok = int(top[n])
                assert lens[b, n] == (0 if tok == 3 else 1) and (tok == 3 or ids[b, n, 0] == tok), (g, b, n)
                assert abs(float(lp[b, n]) - tf[b, tok]) <= 2e-3, (g, b, n)
        print("G=%d: %d of %d images separated enough to check" % (g, checked, B))
        assert checked >= B // 2
    eng.close()


def test_bit_identical_across_modes_and_engine_settings(subject):
    s = subject
    outs = []
    for kw in (dict(), dict(use_graphs=False), dict(cache_mode="physical"), dict(opts=("no_kv_share",)),
               dict(true_beam=True, finished_beams=True, length_penalty=0.6), dict(finished_beams=True)):
        eng = _engine(s, **kw)
        _load_memory(eng, s)
        for es in (True, False, True):
            outs.append(_search(eng, length_penalty=0.8, early_stop=es, beam_groups=4, diversity=0.5))
        assert _groups_identical(_search(eng, beam_groups=2, diversity=0.0), 2), kw
        eng.close()
    for o in outs[1:]:
        for a, b in zip(o, outs[0]):
            assert np.array_equal(a, b)
    assert (outs[0][1] < T).all(1).any()                          # early stop had something to stop


@pytest.mark.parametrize("cache_mode", ["ancestry", "physical"])
def test_diverse_search_leaves_other_decodes_and_launch_count_unchanged(subject, cache_mode):
    s = subject
    eng = _engine(s, cache_mode=cache_mode)
    c0 = eng.launch_count
    g0 = [x.clone() for x in eng.generate(s["img"], early_stop=False)]
    c1 = eng.launch_count
    s0 = [x.clone() for x in eng.sample(None, temperature=0.9, top_k=20, seed=3, return_logprobs=True)]
    ids, lens = s0[0].numpy(), s0[1].numpy()
    sc0 = _score(eng, ids, lens)
    b0 = _search(eng, length_penalty=0.8)
    _search(eng, length_penalty=0.8, beam_groups=4, diversity=0.5)
    _search(eng, s["img"], length_penalty=0.0, early_stop=False, beam_groups=8, diversity=2.0)
    c2 = eng.launch_count
    g1 = eng.generate(s["img"], early_stop=False)
    c3 = eng.launch_count
    s1 = eng.sample(None, temperature=0.9, top_k=20, seed=3, return_logprobs=True)
    sc1 = _score(eng, ids, lens)
    b1 = _search(eng, length_penalty=0.8)
    eng.close()
    assert c3 - c2 == c1 - c0
    for a, b in zip(g0 + s0, list(g1) + list(s1)):
        assert torch.equal(a, b)
    assert np.array_equal(sc0, sc1)
    for a, b in zip(b0, b1):
        assert np.array_equal(a, b)


def test_errors_dlpack_and_pipeline(subject):
    from fpnmt import _lib
    from fpnmt._lib import FpnmtError
    s = subject
    for kw in (dict(decode_path="fused"), dict(score_mode="prob")):
        e = _engine(s, **kw)
        with pytest.raises(FpnmtError) as ei:
            e.beam_search(s["img"], beam_groups=2, diversity=0.5)
        assert ei.value.code == _lib.ERR_STATE, kw
        e.close()
    eng = _engine(s)
    _load_memory(eng, s)
    c0 = eng.launch_count
    for g, lam, alpha in ((0, 0.5, 0.0), (-2, 0.5, 0.0), (3, 0.5, 0.0), (16, 0.5, 0.0), (2, -0.5, 0.0), (2, float("nan"), 0.0),
                          (2, float("inf"), 0.0), (2, 0.5, float("nan")), (2, 0.5, float("inf"))):
        with pytest.raises(FpnmtError) as ei:
            eng.beam_search(None, beam_groups=g, diversity=lam, length_penalty=alpha)
        assert ei.value.code == _lib.ERR_INVALID, (g, lam, alpha)
    assert eng.launch_count == c0                                 # nothing launched
    stream = torch.cuda.current_stream().cuda_stream
    ids = torch.zeros((B, N, T), dtype=torch.int32, device="cuda")
    lens = torch.zeros((B, N), dtype=torch.int32, device="cuda")
    lp = torch.zeros((B, N), dtype=torch.float32, device="cuda")
    f = eng.lib.fpnmt_beam_search_diverse
    assert f(eng._h, None, 0, 2, C.c_float(0.5), C.c_float(0.0), None, lens.data_ptr(), None, 0, 1, stream) == _lib.ERR_INVALID
    assert f(eng._h, None, 0, 2, C.c_float(0.5), C.c_float(0.0), ids.data_ptr(), None, None, 0, 1, stream) == _lib.ERR_INVALID
    # DLPack twin == pointer entry point
    ref = eng.beam_search(None, length_penalty=0.5, beam_groups=4, diversity=0.5, to_host=False, return_logprobs=True)
    keep = []

    def dl(x):
        p, k = _lib.dl_tensor(x)
        keep.append(k)
        return p
    assert eng.lib.fpnmt_beam_search_diverse_dl(eng._h, None, 4, C.c_float(0.5), C.c_float(0.5), dl(ids), dl(lens), dl(lp), 1,
                                                stream) == 0
    torch.cuda.synchronize()
    assert torch.equal(ids, ref[0]) and torch.equal(lens, ref[1]) and torch.equal(lp, ref[2])
    bad_ids = torch.zeros((B, N, T + 1), dtype=torch.int32, device="cuda")
    assert eng.lib.fpnmt_beam_search_diverse_dl(eng._h, None, 4, C.c_float(0.5), C.c_float(0.5), dl(bad_ids), dl(lens), None,
                                                1, stream) == _lib.ERR_INVALID
    assert eng.lib.fpnmt_beam_search_diverse_dl(eng._h, None, 3, C.c_float(0.5), C.c_float(0.5), dl(ids), dl(lens), None, 1,
                                                stream) == _lib.ERR_INVALID
    eng.close()
    # lane 0 holding a submitted batch
    lanes = _engine(s, lanes=2)
    keep_img = lanes.submit(0, s["img"].cuda(), early_stop=False)
    with pytest.raises(FpnmtError) as ei:
        lanes.beam_search(None, beam_groups=2, diversity=0.5)
    assert ei.value.code == _lib.ERR_STATE
    lanes.collect(0)
    del keep_img
    lanes.close()
    # Pipeline.beam_search_batch runs the cached engine's diverse search
    from fpnmt.dataset import Tokenizer
    from fpnmt.pipeline import Pipeline
    w = O.caption_weights(BB, vocab=512, layers=6, seed=0, end_bias=END_BIAS)
    img = O.test_images(2, 512, seed=41)
    pipe = Pipeline(None, None, 12, tokenizer=Tokenizer.synthetic(512), weights=w, beam=4, precision="bf16")
    out = pipe.beam_search_batch(img, 12, num_beams=6, length_penalty=0.8, return_logprobs=True, beam_groups=3, diversity=0.5)
    ref = pipe.transformer.engine(2, 6, 12).beam_search(img, length_penalty=0.8, return_logprobs=True, beam_groups=3,
                                                        diversity=0.5)
    assert out[0].shape == (2, 6, 12) and out[1].shape == (2, 6) and out[2].shape == (2, 6)
    for a, b in zip(out, ref):
        assert np.array_equal(a, b.numpy())
