"""N-best beam search (Engine.beam_search / fpnmt_beam_search, Pipeline.beam_search_batch) against the oracle
(tests/beam_search_oracle.py), against `score` and against itself.

Subject: the sizes of test_gpu_beam_ext.py (S = 256, L = 2, V = 1000, T = 16, N = 8, B = 24) with an <end> bias that ends
about half of the beams before T, so lists hold finished and truncated captions and some images close before the last step.

Bounds (absolute, per scored position n = min(len + 1, T)):
  bf16x3  2e-3: the per-term bound of test_gpu_scoring.py.  A list counts as identical when all N ids and lens match; >= 90 %
          of the images must (the N-best list is N fragile rankings, not one: a 1-ulp difference of the two length-penalty
          tables, powf on the host against numpy, or a near-tie of two candidates' bf16x3 scores may reorder it).
  bf16    0.25: the per-caption bound of test_gpu_scoring.py, against the fp64 teacher-forced sum of the returned caption,
          and between the beam score and `score` of the same caption.
Exact (bit-equal): early stop on / off, graphs on / off, two runs, ancestry / physical cache, default / no_kv_share, engines
created with other true_beam / finished_beams / length_penalty settings; row 0 at alpha = 0 against generate on a
true_beam + finished_beams engine; generate / sample / score and generate's launch count after a beam search.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import fpnmt_oracle as O
import beam_search_oracle as BO

pytestmark = pytest.mark.gpu

BB, S, L, V, T, N, B = "mobilenet224_1.0", 256, 2, 1000, 16, 8, 24
END_BIAS = 12.0


@pytest.fixture(scope="module")
def subject():
    w = O.caption_weights(BB, vocab=V, layers=L, seed=0, end_bias=END_BIAS)
    Wv = O.W(w)
    img = O.test_images(B, S, seed=41)
    with torch.no_grad():
        mem = O.encoder(img, Wv, BB, num_layers=L, input_vocab_size=(S // 16) ** 2)
    return dict(w=w, Wv=Wv, W64=O.W(w, torch.float64), img=img, mem=mem)


def _engine(s, prec="bf16", **kw):
    from fpnmt.engine import Engine
    return Engine(s["w"], backbone=BB, batch=B, beam=N, vocab=V, max_len=T, num_layers=L, image_size=S, precision=prec, **kw)


def _load_memory(eng, s):
    eng.decode_logits(s["mem"].cuda(), torch.full((B, 1), 2, dtype=torch.int32).cuda())


def _search(eng, images=None, **kw):
    return [x.clone().numpy() for x in eng.beam_search(images, return_logprobs=True, **kw)]


def _n(lens):
    return np.minimum(lens + 1, T)


def _check_structure(ids, lens, lp, alpha):
    table = BO.length_penalty_table(T, alpha)
    assert ((lens >= 0) & (lens <= T)).all()
    key = lp.astype(np.float64) / table[_n(lens)]
    # rank order (equal keys: slot order); the engine's table comes from powf, this one from numpy: 1 ulp of slack
    assert (key[:, :-1] >= key[:, 1:] - 2.0 ** -22 * np.abs(key[:, 1:])).all()
    for b in range(B):
        caps = [tuple(ids[b, n, :lens[b, n]]) for n in range(N)]
        assert len(set(caps)) == N, b
        assert all(3 not in c for c in caps), b
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


@pytest.mark.parametrize("alpha", [0.0, 0.8])
def test_bf16x3_matches_oracle_and_score(subject, alpha):
    s = subject
    ref_ids, ref_len, ref_lp = BO.beam_search_nbest(s["mem"], s["Wv"], T, N, 2, 3, length_penalty=alpha, num_layers=L)
    assert (ref_len < T).sum() >= 20 and (ref_len == T).sum() >= 20 and (ref_len < T).all(1).any()
    eng = _engine(s, "bf16x3")
    _load_memory(eng, s)
    ids, lens, lp = _search(eng, length_penalty=alpha)
    sc = _score(eng, ids, lens)                                   # the memory the search left
    eng.close()
    _check_structure(ids, lens, lp, alpha)
    same = (ids == ref_ids).all(axis=(1, 2)) & (lens == ref_len).all(axis=1)
    err = (np.abs(lp - ref_lp) / _n(lens))[same]
    print("bf16x3 alpha=%g: %d / %d N-best lists identical to the oracle, worst |dlogprob| / n %.2e, "
          "worst |score - logprob| / n %.2e" % (alpha, same.sum(), B, err.max(), (np.abs(sc - lp) / _n(lens)).max()))
    assert same.mean() >= 0.9
    assert err.max() <= 2e-3
    assert (np.abs(sc - lp) <= 2e-3 * _n(lens)).all()


@pytest.mark.parametrize("opts", [(), ("tgemm_wide",)])
def test_bf16_structure_likelihood_and_score(subject, opts):
    s = subject
    eng = _engine(s, opts=opts)
    _load_memory(eng, s)
    for alpha in (0.0, 0.8):
        ids, lens, lp = _search(eng, length_penalty=alpha)
        sc = _score(eng, ids, lens)
        _check_structure(ids, lens, lp, alpha)
        assert (lens < T).any() and (lens == T).any()
        ref = _teacher_forced_sum(s, ids, lens)
        e_ref = np.abs(lp - ref) / _n(lens)
        e_sc = np.abs(sc - lp) / _n(lens)
        print("bf16 %s alpha=%g: worst |logprob - fp64| / n %.3f, worst |score - logprob| / n %.3f"
              % (opts, alpha, e_ref.max(), e_sc.max()))
        assert e_ref.max() <= 0.25 and e_sc.max() <= 0.25
    eng.close()


def test_bit_identical_across_modes_and_engine_settings(subject):
    s = subject
    outs = []
    for kw in (dict(), dict(use_graphs=False), dict(cache_mode="physical"), dict(opts=("no_kv_share",)),
               dict(true_beam=True, finished_beams=True, length_penalty=0.6), dict(finished_beams=True)):
        eng = _engine(s, **kw)
        _load_memory(eng, s)
        for es in (True, False, True):
            outs.append(_search(eng, length_penalty=0.8, early_stop=es))
        eng.close()
    for o in outs[1:]:
        for a, b in zip(o, outs[0]):
            assert np.array_equal(a, b)
    assert (outs[0][1] < T).all(1).any()                          # early stop had something to stop


def test_row0_equals_generate_of_a_finished_beams_engine(subject):
    s = subject
    eng = _engine(s, true_beam=True, finished_beams=True)
    g_ids, g_len = eng.generate(s["img"], early_stop=True)
    ids, lens, _ = _search(eng, length_penalty=0.0)
    ids2, lens2, _ = _search(eng, s["img"], length_penalty=0.0)
    eng.close()
    assert np.array_equal(ids[:, 0], g_ids.numpy()) and np.array_equal(lens[:, 0], g_len.numpy())
    assert np.array_equal(ids, ids2) and np.array_equal(lens, lens2)


@pytest.mark.parametrize("cache_mode", ["ancestry", "physical"])
def test_beam_search_leaves_generate_sample_score_and_launch_count_unchanged(subject, cache_mode):
    s = subject
    eng = _engine(s, cache_mode=cache_mode)
    c0 = eng.launch_count
    g0 = [x.clone() for x in eng.generate(s["img"], early_stop=False)]
    c1 = eng.launch_count
    s0 = [x.clone() for x in eng.sample(None, temperature=0.9, top_k=20, seed=3, return_logprobs=True)]
    ids, lens = s0[0].numpy(), s0[1].numpy()
    sc0 = _score(eng, ids, lens)
    _search(eng, length_penalty=0.8)
    _search(eng, s["img"], length_penalty=0.0, early_stop=False)
    c2 = eng.launch_count
    g1 = eng.generate(s["img"], early_stop=False)
    c3 = eng.launch_count
    s1 = eng.sample(None, temperature=0.9, top_k=20, seed=3, return_logprobs=True)
    sc1 = _score(eng, ids, lens)
    eng.close()
    assert c3 - c2 == c1 - c0
    for a, b in zip(g0 + s0, list(g1) + list(s1)):
        assert torch.equal(a, b)
    assert np.array_equal(sc0, sc1)


def test_errors_dlpack_and_pipeline(subject):
    from fpnmt import _lib
    from fpnmt._lib import FpnmtError
    s = subject
    for kw in (dict(decode_path="fused"), dict(score_mode="prob")):
        e = _engine(s, **kw)
        with pytest.raises(FpnmtError) as ei:
            e.beam_search(s["img"])
        assert ei.value.code == _lib.ERR_STATE, kw
        e.close()
    eng = _engine(s)
    _load_memory(eng, s)
    for bad in (float("nan"), float("inf")):
        with pytest.raises(FpnmtError) as ei:
            eng.beam_search(None, length_penalty=bad)
        assert ei.value.code == _lib.ERR_INVALID, bad
    stream = torch.cuda.current_stream().cuda_stream
    ids = torch.zeros((B, N, T), dtype=torch.int32, device="cuda")
    lens = torch.zeros((B, N), dtype=torch.int32, device="cuda")
    lp = torch.zeros((B, N), dtype=torch.float32, device="cuda")
    assert eng.lib.fpnmt_beam_search(eng._h, None, 0, C.c_float(0.0), None, lens.data_ptr(), None, 0, 1, stream) == _lib.ERR_INVALID
    assert eng.lib.fpnmt_beam_search(eng._h, None, 0, C.c_float(0.0), ids.data_ptr(), None, None, 0, 1, stream) == _lib.ERR_INVALID
    # DLPack twin == pointer entry point
    ref = eng.beam_search(None, length_penalty=0.5, to_host=False, return_logprobs=True)
    keep = []

    def dl(x):
        p, k = _lib.dl_tensor(x)
        keep.append(k)
        return p
    assert eng.lib.fpnmt_beam_search_dl(eng._h, None, C.c_float(0.5), dl(ids), dl(lens), dl(lp), 1, stream) == 0
    torch.cuda.synchronize()
    assert torch.equal(ids, ref[0]) and torch.equal(lens, ref[1]) and torch.equal(lp, ref[2])
    bad_ids = torch.zeros((B, N, T + 1), dtype=torch.int32, device="cuda")
    assert eng.lib.fpnmt_beam_search_dl(eng._h, None, C.c_float(0.5), dl(bad_ids), dl(lens), None, 1, stream) == _lib.ERR_INVALID
    eng.close()
    # lane 0 holding a submitted batch
    lanes = _engine(s, lanes=2)
    keep_img = lanes.submit(0, s["img"].cuda(), early_stop=False)
    with pytest.raises(FpnmtError) as ei:
        lanes.beam_search(None)
    assert ei.value.code == _lib.ERR_STATE
    lanes.collect(0)
    del keep_img
    lanes.close()
    # Pipeline.beam_search_batch runs the cached engine's beam_search
    from fpnmt.dataset import Tokenizer
    from fpnmt.pipeline import Pipeline
    w = O.caption_weights(BB, vocab=512, layers=6, seed=0, end_bias=END_BIAS)
    img = O.test_images(2, 512, seed=41)
    pipe = Pipeline(None, None, 12, tokenizer=Tokenizer.synthetic(512), weights=w, beam=4, precision="bf16")
    out = pipe.beam_search_batch(img, 12, num_beams=6, length_penalty=0.8, return_logprobs=True)
    ref = pipe.transformer.engine(2, 6, 12).beam_search(img, length_penalty=0.8, return_logprobs=True)
    assert out[0].shape == (2, 6, 12) and out[1].shape == (2, 6) and out[2].shape == (2, 6)
    for a, b in zip(out, ref):
        assert np.array_equal(a, b.numpy())
