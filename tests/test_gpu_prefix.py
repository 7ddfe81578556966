"""Prompted decoding (Engine.beam_search / Engine.sample with prefix, fpnmt_beam_search_prefix / fpnmt_sample_prefix,
Pipeline.beam_search_batch(prefix=...)) against the oracle (tests/prefix_oracle.py), against `score` and against the
unprompted calls; and the target epilogue of the vocabulary projection (fpnmt_op_vocab_stats_target) one kernel at a time.

Subject: that of test_gpu_beam_search.py (S 256, L 2, V 1000, T 16, N 8, B 24, <end> bias 12), prefixes of random tokens with
lengths 0 .. 5 mixed across images (prefix_len[b] = b % 6).

Bounds (absolute, per scored position n = min(len + 1, T)), those of test_gpu_beam_search.py / test_gpu_sampling.py:
  bf16x3  2e-3; >= 90 % of the N-best lists and >= 95 % of the samples identical to the oracle.
  bf16    0.25 against the fp64 teacher-forced sum of the returned caption and between the beam score and `score`.
Exact (bit-equal): all prefix_len = 0 against the unprompted call (N-best, diverse G = 2 and sampling; logits and logits-free
tails, graphs on / off, both cache modes, no_kv_share); early stop on / off and two runs; other images under a changed or an
invalid prefix; sampling / greedy with a sample's own first k tokens; generate / sample / score and generate's launch count
after a prompted call.
Target epilogue: exact inputs (x = a/8, W = b/16, bias a multiple of 1/128: every logit is an fp32 number) give the logit
bit for bit; random inputs are within the fp32-accumulation bound of test_gpu_vocab_tail.py, K 2^-23 sum |x w| + 2^-24 |z|,
of the fp64 logit of the bf16-rounded operands, and bit-equal to the tile's candidate value wherever the target is one.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import fpnmt_oracle as O
import beam_search_oracle as BO
import prefix_oracle as PO

pytestmark = pytest.mark.gpu

BB, S, L, V, T, N, B = "mobilenet224_1.0", 256, 2, 1000, 16, 8, 24
END_BIAS = 12.0
P = 5


@pytest.fixture(scope="module")
def subject():
    w = O.caption_weights(BB, vocab=V, layers=L, seed=0, end_bias=END_BIAS)
    Wv = O.W(w)
    img = O.test_images(B, S, seed=41)
    with torch.no_grad():
        mem = O.encoder(img, Wv, BB, num_layers=L, input_vocab_size=(S // 16) ** 2)
    rng = np.random.default_rng(3)
    prefix = rng.integers(4, V, size=(B, P)).astype(np.int32)
    plen = (np.arange(B) % 6).astype(np.int32)
    return dict(w=w, Wv=Wv, W64=O.W(w, torch.float64), img=img, mem=mem, prefix=prefix, plen=plen)


def _engine(s, prec="bf16", **kw):
    from fpnmt.engine import Engine
    return Engine(s["w"], backbone=BB, batch=B, beam=N, vocab=V, max_len=T, num_layers=L, image_size=S, precision=prec, **kw)


def _load_memory(eng, s):
    eng.decode_logits(s["mem"].cuda(), torch.full((B, 1), 2, dtype=torch.int32).cuda())


def _search(eng, images=None, **kw):
    return [x.clone().numpy() for x in eng.beam_search(images, return_logprobs=True, **kw)]


def _sample(eng, images=None, **kw):
    return [x.clone().numpy() for x in eng.sample(images, return_logprobs=True, **kw)]


SAMPLING = dict(temperature=0.9, top_k=20, top_p=0.95, seed=11)


def _n(lens):
    return np.minimum(lens + 1, T)


def _check_prefix(s, ids, lens, prefix=None, plen=None):
    prefix = s["prefix"] if prefix is None else prefix
    plen = s["plen"] if plen is None else plen
    for b in range(B):
        k = int(plen[b])
        assert (lens[b] >= k).all(), b
        assert (ids[b, :, :k] == prefix[b, :k]).all(), b
    assert not (ids * (np.arange(T)[None, None, :] >= lens[..., None])).any()   # zero past len


def _check_structure(ids, lens, lp, alpha, groups=1):
    table = BO.length_penalty_table(T, alpha)
    key = lp.astype(np.float64) / table[_n(lens)]
    m = N // groups
    for g in range(groups):
        k = key[:, g * m:(g + 1) * m]
        assert (k[:, :-1] >= k[:, 1:] - 2.0 ** -22 * np.abs(k[:, 1:])).all()
        for b in range(B):
            caps = [tuple(ids[b, n, :lens[b, n]]) for n in range(g * m, (g + 1) * m)]
            assert len(set(caps)) == m, b
            assert all(3 not in c for c in caps), b
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


def _pfx(s, **kw):
    return dict(prefix=s["prefix"], prefix_lens=s["plen"], **kw)


# ---------------------------------------------------------------------------------------------------------------------------
def test_bf16x3_matches_oracle_and_score(subject):
    s = subject
    ref_ids, ref_len, ref_lp = PO.prefix_beam_search(s["mem"], s["Wv"], T, N, 1, 0.0, 2, 3, s["prefix"], s["plen"],
                                                     length_penalty=0.8, num_layers=L)
    ref_s = PO.prefix_sample(s["mem"], s["Wv"], T, N, 2, 3, s["prefix"], s["plen"], num_layers=L, **SAMPLING)
    eng = _engine(s, "bf16x3")
    _load_memory(eng, s)
    ids, lens, lp = _search(eng, **_pfx(s, length_penalty=0.8))
    sc = _score(eng, ids, lens)
    sids, slens, slp = _sample(eng, **_pfx(s, **SAMPLING))
    eng.close()
    _check_prefix(s, ids, lens)
    _check_structure(ids, lens, lp, 0.8)
    same = (ids == ref_ids).all(axis=(1, 2)) & (lens == ref_len).all(axis=1)
    err = (np.abs(lp - ref_lp) / _n(lens))[same]
    print("bf16x3: %d / %d prompted N-best lists identical to the oracle, worst |dlogprob| / n %.2e" % (same.sum(), B, err.max()))
    assert same.mean() >= 0.9
    assert err.max() <= 2e-3
    assert (np.abs(sc - lp) <= 2e-3 * _n(lens)).all()
    _check_prefix(s, sids, slens)
    ssame = (sids == ref_s[0]).all(-1) & (slens == ref_s[1])
    print("bf16x3: %d / %d prompted samples identical to the oracle" % (ssame.sum(), ssame.size))
    assert ssame.mean() >= 0.95
    assert float((np.abs(slp - ref_s[2])[ssame] / (slens[ssame] + 1)).max()) <= 2e-3


@pytest.mark.parametrize("opts", [(), ("tgemm_wide",)])
def test_bf16_structure_likelihood_and_score(subject, opts):
    s = subject
    eng = _engine(s, opts=opts)
    _load_memory(eng, s)
    for g, lam in ((1, 0.0), (2, 0.5)):
        ids, lens, lp = _search(eng, **_pfx(s, length_penalty=0.8, beam_groups=g, diversity=lam))
        sc = _score(eng, ids, lens)
        _check_prefix(s, ids, lens)
        _check_structure(ids, lens, lp, 0.8, g)
        ref = _teacher_forced_sum(s, ids, lens)
        e_ref, e_sc = np.abs(lp - ref) / _n(lens), np.abs(sc - lp) / _n(lens)
        print("bf16 %s G=%d: worst |logprob - fp64| / n %.3f, |score - logprob| / n %.3f" % (opts, g, e_ref.max(), e_sc.max()))
        assert e_ref.max() <= 0.25 and e_sc.max() <= 0.25
    sids, slens, slp = _sample(eng, **_pfx(s, **SAMPLING))
    _check_prefix(s, sids, slens)
    ref = _teacher_forced_sum(s, sids, slens)
    assert (np.abs(slp - ref) / _n(slens)).max() <= 0.25
    eng.close()


@pytest.mark.parametrize("kw", [dict(), dict(use_graphs=False), dict(cache_mode="physical"), dict(opts=("no_kv_share",)),
                                dict(opts=("tgemm_wide",)), dict(opts=("tgemm_wide",), cache_mode="physical", use_graphs=False)])
def test_empty_prefixes_are_the_unprompted_calls(subject, kw):
    s = subject
    eng = _engine(s, **kw)
    _load_memory(eng, s)
    zero = dict(prefix=s["prefix"], prefix_lens=np.zeros(B, np.int32))
    for call, args in ((_search, dict(length_penalty=0.8)), (_search, dict(length_penalty=0.8, beam_groups=2, diversity=0.5)),
                       (_sample, SAMPLING)):
        a = call(eng, **args)
        b = call(eng, **args, **zero)
        for x, y in zip(a, b):
            assert np.array_equal(x, y), (kw, args)
    eng.close()


@pytest.mark.parametrize("opts", [(), ("tgemm_wide",)])
def test_bit_exact_early_stop_runs_other_images_and_invalid_prefixes(subject, opts):
    s = subject
    eng = _engine(s, opts=opts)
    _load_memory(eng, s)
    for call, args in ((_search, dict(length_penalty=0.8)), (_search, dict(beam_groups=2, diversity=0.5)), (_sample, SAMPLING)):
        ref = call(eng, **_pfx(s, **args))
        for es in (False, True):
            for x, y in zip(ref, call(eng, early_stop=es, **_pfx(s, **args))):
                assert np.array_equal(x, y), (opts, args, es)
        # one image's prefix changed: every other image's result stays
        pf, pl = s["prefix"].copy(), s["plen"].copy()
        pf[7] = (pf[7] + 13) % (V - 4) + 4
        pl[7] = 4
        other = call(eng, prefix=pf, prefix_lens=pl, **args)
        keep = np.arange(B) != 7
        for x, y in zip(ref, other):
            assert np.array_equal(x[keep], y[keep]), (opts, args)
        _check_prefix(s, other[0], other[1], pf, pl)
        # invalid images: len outside [0, p], an id out of range, <end> inside the prefix
        pf, pl = s["prefix"].copy(), s["plen"].copy()
        pl[2], pl[3] = P + 1, -1
        pl[4], pf[4, 1] = 3, V
        pl[5], pf[5, 0] = 2, 3
        pf[8, 4] = -5                                               # beyond image 8's prefix length (2): ignored, still valid
        bad = np.isin(np.arange(B), [2, 3, 4, 5])
        got = call(eng, prefix=pf, prefix_lens=pl, **args)
        for x, y in zip(ref, got):
            assert np.array_equal(x[~bad], y[~bad]), (opts, args)
        assert (got[0][bad] == 0).all() and (got[1][bad] == 0).all() and np.isnan(got[2][bad]).all()
    eng.close()


def test_own_prefix_reproduces_the_sample_and_greedy(subject):
    s = subject
    eng = _engine(s)
    _load_memory(eng, s)
    for args in (SAMPLING, dict(temperature=0.0)):
        ids, lens, lp = _sample(eng, **args)
        for k in range(1, 5):
            ok = lens[:, 0] >= k
            pf = np.zeros((B, k), np.int32)
            pf[ok] = ids[ok, 0, :k]
            got = _sample(eng, prefix=pf, prefix_lens=np.where(ok, k, 0).astype(np.int32), **args)
            assert ok.sum() >= B // 2
            for x, y in zip((ids, lens, lp), got):
                assert np.array_equal(x[:, 0], y[:, 0]), (args, k)
                assert np.array_equal(x[~ok], y[~ok]), (args, k)
    eng.close()


def test_one_group_is_the_nbest_prompted_search(subject):
    s = subject
    eng = _engine(s, opts=("tgemm_wide",))
    _load_memory(eng, s)
    a = _search(eng, **_pfx(s, length_penalty=0.8))
    b = _search(eng, **_pfx(s, length_penalty=0.8, beam_groups=1, diversity=0.7))
    eng.close()
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


@pytest.mark.parametrize("kw", [dict(), dict(cache_mode="physical", opts=("tgemm_wide",))])
def test_prompted_calls_leave_generate_sample_score_and_launch_count_unchanged(subject, kw):
    s = subject
    eng = _engine(s, **kw)
    c0 = eng.launch_count
    g0 = [x.clone() for x in eng.generate(s["img"], early_stop=False)]
    c1 = eng.launch_count
    s0 = [x.clone() for x in eng.sample(None, return_logprobs=True, **SAMPLING)]
    ids, lens = s0[0].numpy(), s0[1].numpy()
    sc0 = _score(eng, ids, lens)
    b0 = _search(eng, length_penalty=0.8)
    _search(eng, **_pfx(s, length_penalty=0.8))
    _sample(eng, s["img"], **_pfx(s, **SAMPLING))
    c2 = eng.launch_count
    g1 = eng.generate(s["img"], early_stop=False)
    c3 = eng.launch_count
    s1 = eng.sample(None, return_logprobs=True, **SAMPLING)
    sc1 = _score(eng, ids, lens)
    b1 = _search(eng, length_penalty=0.8)
    eng.close()
    assert c3 - c2 == c1 - c0
    for a, b in zip(g0 + s0, list(g1) + list(s1)):
        assert torch.equal(a, b)
    assert np.array_equal(sc0, sc1)
    for x, y in zip(b0, b1):
        assert np.array_equal(x, y)


def test_errors_dlpack_and_pipeline(subject):
    from fpnmt import _lib
    from fpnmt._lib import FpnmtError
    s = subject
    for kw, calls in ((dict(decode_path="fused"), ("beam", "sample")), (dict(score_mode="prob"), ("beam",))):
        e = _engine(s, **kw)
        for c in calls:
            with pytest.raises(FpnmtError) as ei:
                (e.beam_search if c == "beam" else e.sample)(s["img"], **_pfx(s))
            assert ei.value.code == _lib.ERR_STATE, (kw, c)
        e.close()
    eng = _engine(s)
    _load_memory(eng, s)
    stream = torch.cuda.current_stream().cuda_stream
    ids = torch.zeros((B, N, T), dtype=torch.int32, device="cuda")
    lens = torch.zeros((B, N), dtype=torch.int32, device="cuda")
    lp = torch.zeros((B, N), dtype=torch.float32, device="cuda")
    pf = torch.from_numpy(s["prefix"]).cuda()
    pl = torch.from_numpy(s["plen"]).cuda()
    wide = torch.zeros((B, T), dtype=torch.int32, device="cuda")
    sp = _lib.sampling(**SAMPLING)
    for p_ids, p_len, p in ((pf, pl, 0), (wide, pl, T), (None, pl, P), (pf, None, P)):
        args = (p_ids.data_ptr() if p_ids is not None else None, p_len.data_ptr() if p_len is not None else None, p)
        assert eng.lib.fpnmt_beam_search_prefix(eng._h, None, 0, *args, 1, C.c_float(0.0), C.c_float(0.0), ids.data_ptr(),
                                                lens.data_ptr(), None, 0, 1, stream) == _lib.ERR_INVALID
        assert eng.lib.fpnmt_sample_prefix(eng._h, None, 0, *args, C.byref(sp), ids.data_ptr(), lens.data_ptr(), None, 0, 1,
                                           stream) == _lib.ERR_INVALID
    assert eng.lib.fpnmt_beam_search_prefix(eng._h, None, 0, pf.data_ptr(), pl.data_ptr(), P, 3, C.c_float(0.0), C.c_float(0.0),
                                            ids.data_ptr(), lens.data_ptr(), None, 0, 1, stream) == _lib.ERR_INVALID
    # DLPack twins == pointer entry points
    keep = []

    def dl(x):
        p, k = _lib.dl_tensor(x)
        keep.append(k)
        return p
    ref = eng.beam_search(None, to_host=False, return_logprobs=True, **_pfx(s, length_penalty=0.5, beam_groups=2, diversity=0.3))
    assert eng.lib.fpnmt_beam_search_prefix_dl(eng._h, None, dl(pf), dl(pl), 2, C.c_float(0.3), C.c_float(0.5), dl(ids), dl(lens),
                                               dl(lp), 1, stream) == 0
    torch.cuda.synchronize()
    assert torch.equal(ids, ref[0]) and torch.equal(lens, ref[1]) and torch.equal(lp, ref[2])
    ref = eng.sample(None, to_host=False, return_logprobs=True, **_pfx(s, **SAMPLING))
    assert eng.lib.fpnmt_sample_prefix_dl(eng._h, None, dl(pf), dl(pl), C.byref(sp), dl(ids), dl(lens), dl(lp), 1, stream) == 0
    torch.cuda.synchronize()
    assert torch.equal(ids, ref[0]) and torch.equal(lens, ref[1]) and torch.equal(lp, ref[2])
    for bad in (pf[:B - 1], wide, pf[:, :0]):
        assert eng.lib.fpnmt_beam_search_prefix_dl(eng._h, None, dl(bad.contiguous()), dl(pl), 1, C.c_float(0.0), C.c_float(0.0),
                                                   dl(ids), dl(lens), None, 1, stream) == _lib.ERR_INVALID
        assert eng.lib.fpnmt_sample_prefix_dl(eng._h, None, dl(bad.contiguous()), dl(pl), C.byref(sp), dl(ids), dl(lens), None, 1,
                                              stream) == _lib.ERR_INVALID
    eng.close()
    # lane 0 holding a submitted batch
    lanes = _engine(s, lanes=2)
    keep_img = lanes.submit(0, s["img"].cuda(), early_stop=False)
    for fn in (lanes.beam_search, lanes.sample):
        with pytest.raises(FpnmtError) as ei:
            fn(None, **_pfx(s))
        assert ei.value.code == _lib.ERR_STATE
    lanes.collect(0)
    del keep_img
    lanes.close()
    # Pipeline.beam_search_batch / sample_batch with prefix strings run the engine on the tokenized prefixes
    from fpnmt.dataset import Tokenizer
    from fpnmt.pipeline import Pipeline
    w = O.caption_weights(BB, vocab=512, layers=6, seed=0, end_bias=END_BIAS)
    img = O.test_images(2, 512, seed=41)
    tok = Tokenizer.synthetic(512)
    pipe = Pipeline(None, None, 12, tokenizer=tok, weights=w, beam=4, precision="bf16")
    words = [k for k, v in sorted(tok.word_index.items(), key=lambda kv: kv[1]) if v >= 4][:6]
    texts = [" ".join(words[:3]), words[4]]
    seqs = tok.texts_to_sequences(texts)
    pids = np.zeros((2, 3), np.int32)
    for i, q in enumerate(seqs):
        pids[i, :len(q)] = q
    plens = np.array([len(q) for q in seqs], np.int32)
    assert plens.tolist() == [3, 1]
    out = pipe.beam_search_batch(img, 12, num_beams=6, length_penalty=0.8, return_logprobs=True, prefix=texts)
    ref = pipe.transformer.engine(2, 6, 12).beam_search(img, length_penalty=0.8, return_logprobs=True, prefix=pids, prefix_lens=plens)
    for a, b in zip(out, ref):
        assert np.array_equal(a, b.numpy())
    assert (out[0][0, :, :3] == pids[0]).all() and (out[0][1, :, :1] == pids[1, :1]).all()
    with pytest.raises(ValueError):
        pipe.beam_search_batch(img, 12, num_beams=6, prefix=[texts[0], "<end>"])
    with pytest.raises(ValueError):
        pipe.sample_batch(img, 3, prefix=[texts[0], texts[1]])      # 3 tokens need max_seq_len > 3


# ---------------------------------------------------------------------------------------------------------------------------
def _op_case(R, K, F, exact, seed):
    rng = np.random.default_rng(seed)
    if exact:
        x = rng.integers(-8, 9, size=(R, K)) / 8.0
        w = rng.integers(-8, 9, size=(K, F)) / 16.0
        bias = rng.integers(-256, 257, size=F) / 128.0
    else:
        x = rng.standard_normal((R, K))
        w = rng.standard_normal((K, F)) / np.sqrt(K)
        bias = rng.standard_normal(F) * 0.1
    return x.astype(np.float32), w.astype(np.float32), bias.astype(np.float32)


def _bf16(a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(torch.bfloat16).double().numpy()


@pytest.mark.parametrize("R,K,F,exact", [(256, 512, 1000, True), (200, 512, 1000, False), (130, 256, 904, False),
                                         (77, 512, 8 * 129, True)])
def test_vocab_stats_target_operator(R, K, F, exact):
    from fpnmt.engine import vocab_stats, vocab_stats_target
    x, w, bias = _op_case(R, K, F, exact, R + F)
    rng = np.random.default_rng(F)
    tgt = rng.integers(0, F, size=R).astype(np.int32)
    tgt[::7] = -1                                                   # none
    tgt[3::11] = F + rng.integers(0, 200, size=tgt[3::11].shape)   # beyond F, in or past the padded last tile
    last0 = (F - 1) // 128 * 128
    tgt[5::13] = rng.integers(last0, F, size=tgt[5::13].shape)     # the padded last tile
    z64 = _bf16(x) @ _bf16(w) + bias.astype(np.float64)[None, :]
    tgt[1::5] = np.argmax(z64[1::5], -1)                            # the row maximum: one of its tile's candidates
    xd = torch.from_numpy(x).cuda()
    st0, va0, ix0 = vocab_stats(xd, w, bias)
    sentinel = torch.full((R,), 12345.0, device="cuda")
    st, va, ix, tl = vocab_stats_target(xd, w, tgt, bias, target_logit=sentinel.clone())
    torch.cuda.synchronize()
    for a, b in ((st0, st), (va0, va), (ix0, ix)):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    tl = tl.cpu().numpy()
    valid = (tgt >= 0) & (tgt < F)
    assert (tl[~valid] == 12345.0).all()
    rows = np.nonzero(valid)[0]
    zt = z64[rows, tgt[rows]]
    if exact:
        assert np.array_equal(tl[rows].astype(np.float64), zt)
    else:
        absprod = np.abs(_bf16(x)) @ np.abs(_bf16(w))
        delta = K * 2.0 ** -23 * absprod[rows, tgt[rows]] + 2.0 ** -24 * np.abs(zt)
        err = np.abs(tl[rows] - zt)
        print("target logit: worst error / bound %.3f" % (err / delta).max())
        assert (err <= delta).all()
    # bit-equal to the tile's candidate value wherever the target is one
    va, ix = va.cpu().numpy(), ix.cpu().numpy()
    hits = 0
    for r in rows:
        t = tgt[r] // 128
        j = np.nonzero(ix[r, t] == tgt[r])[0]
        if len(j):
            hits += 1
            assert va[r, t, j[0]].view(np.int32) == np.float32(tl[r]).view(np.int32), r
    print("target among its tile's candidates in %d rows" % hits)
    assert hits >= R // 5
