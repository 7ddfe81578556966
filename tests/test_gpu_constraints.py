"""Constrained decoding (Engine.beam_search / Engine.sample with no_repeat_ngram / min_len / banned,
fpnmt_beam_search_constrained / fpnmt_sample_constrained, Pipeline.*_batch(banned_words=...)) against the oracle
(tests/constraint_oracle.py), against `score` and against the unconstrained and prompted calls; and the two operators
(fpnmt_op_vocab_stats_mask, fpnmt_op_ban_mask) one kernel at a time.

Subject and bounds: those of test_gpu_prefix.py (S 256, L 2, V 1000, T 16, N 8, B 24, <end> bias 12, prefix_len[b] = b % 6).
  bf16x3  >= 90 % of the N-best lists and >= 95 % of the samples identical to the oracle.
  bf16    0.25 per scored position against the fp64 teacher-forced sum and between the beam score and `score`.
Structure (every returned caption, both precisions): no banned id, no n-gram ending at or after the prefix that occurs earlier,
len >= min_len, the prefix kept.  Exact (bit-equal): all-off constraints against the unconstrained and the prompted calls
(N-best, diverse G = 2, sampling, greedy; logits and logits-free tails, graphs on / off, both cache modes, no_kv_share).
"""
import ctypes as C

import numpy as np
import pytest
import torch

import fpnmt_oracle as O
import constraint_oracle as CO

pytestmark = pytest.mark.gpu

BB, S, L, V, T, N, B = "mobilenet224_1.0", 256, 2, 1000, 16, 8, 24
END_BIAS = 12.0
P = 5
SAMPLING = dict(temperature=0.9, top_k=20, top_p=0.95, seed=11)
CON = dict(no_repeat_ngram=2, min_len=5)


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
    s = dict(w=w, Wv=Wv, W64=O.W(w, torch.float64), img=img, mem=mem, prefix=prefix, plen=plen)
    # banned: the padding id, <start>, and the three tokens the unconstrained engine emits most; step0: every tile maximum of
    # every image's first logits (each tile's best logit is banned at step 0: the tau trap of the logits-free tail)
    eng = _engine(s)
    lg = _load_memory(eng, s)
    ids, lens, _ = _search(eng, length_penalty=0.8)
    eng.close()
    toks = np.concatenate([ids[b, n, :lens[b, n]] for b in range(B) for n in range(N)])
    s["banned"] = [0, 2] + [int(x) for x in np.argsort(-np.bincount(toks, minlength=V), kind="stable")[:3]]
    z0 = np.pad(lg, ((0, 0), (0, 1024 - V)), constant_values=-np.inf).reshape(B, 8, 128)
    tm = (np.arange(8) * 128)[None, :] + z0.argmax(-1)
    s["step0"] = sorted(set(int(x) for x in tm.ravel()) - {3})
    return s


def _engine(s, prec="bf16", **kw):
    from fpnmt.engine import Engine
    return Engine(s["w"], backbone=BB, batch=B, beam=N, vocab=V, max_len=T, num_layers=L, image_size=S, precision=prec, **kw)


def _load_memory(eng, s):
    return eng.decode_logits(s["mem"].cuda(), torch.full((B, 1), 2, dtype=torch.int32).cuda()).float().cpu().numpy()[:, 0]


def _search(eng, images=None, **kw):
    return [x.clone().numpy() for x in eng.beam_search(images, return_logprobs=True, **kw)]


def _sample(eng, images=None, **kw):
    return [x.clone().numpy() for x in eng.sample(images, return_logprobs=True, **kw)]


def _pfx(s, **kw):
    return dict(prefix=s["prefix"], prefix_lens=s["plen"], **kw)


def _raw(eng, kind, con=None, prefix=None, plen=None, groups=1, diversity=0.0, alpha=0.0, sampling=None):
    """The constrained C entry point itself (all-off constraints included): (rc, [ids, lens, logprob])."""
    from fpnmt import _lib
    ids = torch.zeros((B, N, T), dtype=torch.int32, device="cuda")
    lens = torch.zeros((B, N), dtype=torch.int32, device="cuda")
    lp = torch.zeros((B, N), dtype=torch.float32, device="cuda")
    c = _lib.constraints(**(con or {}))
    pf = torch.from_numpy(prefix).cuda() if prefix is not None else None
    pl = torch.from_numpy(plen).cuda() if plen is not None else None
    pa = (pf.data_ptr() if pf is not None else None, pl.data_ptr() if pl is not None else None,
          int(prefix.shape[1]) if prefix is not None else 0)
    stream = torch.cuda.current_stream().cuda_stream
    if kind == "beam":
        rc = eng.lib.fpnmt_beam_search_constrained(eng._h, None, 0, *pa, groups, C.c_float(diversity), C.c_float(alpha),
                                                   C.byref(c), ids.data_ptr(), lens.data_ptr(), lp.data_ptr(), 0, 1, stream)
    else:
        sp = _lib.sampling(**(sampling or SAMPLING))
        rc = eng.lib.fpnmt_sample_constrained(eng._h, None, 0, *pa, C.byref(sp), C.byref(c), ids.data_ptr(), lens.data_ptr(),
                                              lp.data_ptr(), 0, 1, stream)
    torch.cuda.synchronize()
    return rc, [ids.cpu().numpy(), lens.cpu().numpy(), lp.cpu().numpy()]


def _n(lens):
    return np.minimum(lens + 1, T)


def _check(s, ids, lens, con, banned, plen=None):
    for b in range(B):
        k = int(plen[b]) if plen is not None else 0
        assert (ids[b, :, :k] == s["prefix"][b, :k]).all(), b
        for n in range(N):
            CO.check_caption(ids[b, n, :lens[b, n]], con.get("no_repeat_ngram", 0), con.get("min_len", 0), banned, k)
    assert not (ids * (np.arange(T)[None, None, :] >= lens[..., None])).any()


def _teacher_forced_sum(s, ids, lens):
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


# ---------------------------------------------------------------------------------------------------------------------------
def test_bf16x3_matches_oracle(subject):
    s = subject
    con = dict(CON, banned=s["banned"])
    ref = CO.constrained_beam_search(s["mem"], s["Wv"], T, N, 1, 0.0, 2, 3, prefix=s["prefix"], prefix_len=s["plen"],
                                     length_penalty=0.8, num_layers=L, **con)
    ref_s = CO.constrained_sample(s["mem"], s["Wv"], T, N, 2, 3, prefix=s["prefix"], prefix_len=s["plen"], num_layers=L,
                                  **con, **SAMPLING)
    eng = _engine(s, "bf16x3")
    _load_memory(eng, s)
    ids, lens, lp = _search(eng, **_pfx(s, length_penalty=0.8), **con)
    sids, slens, slp = _sample(eng, **_pfx(s, **SAMPLING), **con)
    eng.close()
    _check(s, ids, lens, CON, s["banned"], s["plen"])
    _check(s, sids, slens, CON, s["banned"], s["plen"])
    same = (ids == ref[0]).all(axis=(1, 2)) & (lens == ref[1]).all(axis=1)
    ssame = (sids == ref_s[0]).all(-1) & (slens == ref_s[1])
    print("bf16x3: %d / %d constrained N-best lists, %d / %d samples identical to the oracle"
          % (same.sum(), B, ssame.sum(), ssame.size))
    assert same.mean() >= 0.9 and ssame.mean() >= 0.95
    assert (np.abs(lp - ref[2]) / _n(lens))[same].max() <= 2e-3


@pytest.mark.parametrize("opts", [(), ("tgemm_wide",)])
def test_bf16_structure_likelihood_and_score(subject, opts):
    s = subject
    eng = _engine(s, opts=opts)
    _load_memory(eng, s)
    cases = [(dict(CON, banned=s["banned"]), True, 1, 0.0), (dict(CON, banned=s["banned"]), False, 2, 0.5),
             (dict(no_repeat_ngram=1, banned=s["step0"]), False, 1, 0.0), (dict(no_repeat_ngram=3, min_len=T), True, 2, 0.5)]
    for con, prompted, g, lam in cases:
        pk = _pfx(s) if prompted else {}
        ids, lens, lp = _search(eng, length_penalty=0.8, beam_groups=g, diversity=lam, **pk, **con)
        _check(s, ids, lens, con, con.get("banned"), s["plen"] if prompted else None)
        sc = _score(eng, ids, lens)
        ref = _teacher_forced_sum(s, ids, lens)
        e_ref, e_sc = np.abs(lp - ref) / _n(lens), np.abs(sc - lp) / _n(lens)
        print("bf16 %s %s G=%d: worst |logprob - fp64| / n %.3f, |score - logprob| / n %.3f"
              % (opts, sorted(con), g, e_ref.max(), e_sc.max()))
        assert e_ref.max() <= 0.25 and e_sc.max() <= 0.25
        for sp in (SAMPLING, dict(temperature=0.0)):
            sids, slens, slp = _sample(eng, **pk, **sp, **con)
            _check(s, sids, slens, con, con.get("banned"), s["plen"] if prompted else None)
            assert (np.abs(slp - _teacher_forced_sum(s, sids, slens)) / _n(slens)).max() <= 0.25
    eng.close()


@pytest.mark.parametrize("kw", [dict(), dict(use_graphs=False), dict(cache_mode="physical"), dict(opts=("no_kv_share",)),
                                dict(opts=("tgemm_wide",)), dict(opts=("tgemm_wide",), cache_mode="physical", use_graphs=False)])
def test_all_off_is_the_unconstrained_and_prompted_calls(subject, kw):
    s = subject
    eng = _engine(s, **kw)
    _load_memory(eng, s)
    for kind, args, raw in (("beam", dict(length_penalty=0.8), dict(alpha=0.8)),
                            ("beam", dict(length_penalty=0.8, beam_groups=2, diversity=0.5), dict(alpha=0.8, groups=2, diversity=0.5)),
                            ("sample", SAMPLING, dict(sampling=SAMPLING)),
                            ("sample", dict(temperature=0.0), dict(sampling=dict(temperature=0.0)))):
        call = _search if kind == "beam" else _sample
        for pk, rk in (({}, {}), (_pfx(s), dict(prefix=s["prefix"], plen=s["plen"]))):
            a = call(eng, **args, **pk)
            rc, b = _raw(eng, kind, **raw, **rk)
            assert rc == 0
            for x, y in zip(a, b):
                assert np.array_equal(x, y), (kw, kind, args, bool(pk))
    eng.close()


@pytest.mark.parametrize("opts", [(), ("tgemm_wide",)])
def test_bit_exact_repeats_early_stop_and_refusals(subject, opts):
    from fpnmt import _lib
    s = subject
    eng = _engine(s, opts=opts)
    _load_memory(eng, s)
    con = dict(CON, banned=s["banned"])
    for call, args in ((_search, dict(length_penalty=0.8)), (_search, dict(beam_groups=2, diversity=0.5)), (_sample, SAMPLING)):
        ref = call(eng, **_pfx(s, **args), **con)
        for es in (False, True):
            for x, y in zip(ref, call(eng, early_stop=es, **_pfx(s, **args), **con)):
                assert np.array_equal(x, y), (opts, args, es)
    bad = [dict(banned=[V]), dict(banned=[-1]), dict(banned=[3]), dict(no_repeat_ngram=T + 1), dict(no_repeat_ngram=-1),
           dict(min_len=T + 1), dict(min_len=-1), dict(banned=list(range(4, 4 + V - T - N + 1)))]
    c0 = eng.launch_count
    for con in bad:
        for kind in ("beam", "sample"):
            assert _raw(eng, kind, con)[0] == _lib.ERR_INVALID, (con, kind)
    c = _lib.constraints(min_len=2)
    c.reserved[1] = 1
    ids = torch.zeros((B, N, T), dtype=torch.int32, device="cuda")
    lens = torch.zeros((B, N), dtype=torch.int32, device="cuda")
    assert eng.lib.fpnmt_beam_search_constrained(eng._h, None, 0, None, None, 0, 1, C.c_float(0.0), C.c_float(0.0), C.byref(c),
                                                 ids.data_ptr(), lens.data_ptr(), None, 0, 1, None) == _lib.ERR_INVALID
    assert eng.launch_count == c0
    # the largest static list the bound allows runs, and keeps every caption inside the allowed ids
    ok = list(range(4, 4 + V - T - N)) + [4, 5]                   # duplicates count once
    rc, (ids, lens, _) = _raw(eng, "beam", dict(banned=ok), alpha=0.8)
    assert rc == 0 and not np.isin(ids[np.arange(T)[None, None, :] < lens[..., None]], ok).any()
    eng.close()


@pytest.mark.parametrize("kw", [dict(), dict(cache_mode="physical", opts=("tgemm_wide",))])
def test_constrained_calls_leave_generate_sample_score_and_launch_count_unchanged(subject, kw):
    s = subject
    eng = _engine(s, **kw)
    c0 = eng.launch_count
    g0 = [x.clone() for x in eng.generate(s["img"], early_stop=False)]
    c1 = eng.launch_count
    s0 = [x.clone() for x in eng.sample(None, return_logprobs=True, **SAMPLING)]
    ids, lens = s0[0].numpy(), s0[1].numpy()
    sc0 = _score(eng, ids, lens)
    b0 = _search(eng, length_penalty=0.8)
    p0 = _search(eng, **_pfx(s, length_penalty=0.8))
    _search(eng, **_pfx(s, length_penalty=0.8), **CON, banned=s["banned"])
    _sample(eng, s["img"], **SAMPLING, **CON, banned=s["banned"])
    c2 = eng.launch_count
    g1 = eng.generate(s["img"], early_stop=False)
    c3 = eng.launch_count
    s1 = eng.sample(None, return_logprobs=True, **SAMPLING)
    sc1 = _score(eng, ids, lens)
    b1 = _search(eng, length_penalty=0.8)
    p1 = _search(eng, **_pfx(s, length_penalty=0.8))
    eng.close()
    assert c3 - c2 == c1 - c0
    for a, b in zip(g0 + s0, list(g1) + list(s1)):
        assert torch.equal(a, b)
    assert np.array_equal(sc0, sc1)
    for x, y in zip(b0 + p0, b1 + p1):
        assert np.array_equal(x, y)


def test_states_dlpack_and_pipeline(subject):
    from fpnmt import _lib
    from fpnmt._lib import FpnmtError
    s = subject
    for kw, calls in ((dict(decode_path="fused"), ("beam", "sample")), (dict(score_mode="prob"), ("beam",))):
        e = _engine(s, **kw)
        for c in calls:
            with pytest.raises(FpnmtError) as ei:
                (e.beam_search if c == "beam" else e.sample)(s["img"], min_len=2)
            assert ei.value.code == _lib.ERR_STATE, (kw, c)
        e.close()
    lanes = _engine(s, lanes=2)
    keep_img = lanes.submit(0, s["img"].cuda(), early_stop=False)
    for fn in (lanes.beam_search, lanes.sample):
        with pytest.raises(FpnmtError) as ei:
            fn(None, banned=[0])
        assert ei.value.code == _lib.ERR_STATE
    lanes.collect(0)
    del keep_img
    lanes.close()
    # DLPack twins == the engine's calls
    eng = _engine(s)
    _load_memory(eng, s)
    keep = []

    def dl(x):
        p, k = _lib.dl_tensor(x)
        keep.append(k)
        return p
    stream = torch.cuda.current_stream().cuda_stream
    ids = torch.zeros((B, N, T), dtype=torch.int32, device="cuda")
    lens = torch.zeros((B, N), dtype=torch.int32, device="cuda")
    lp = torch.zeros((B, N), dtype=torch.float32, device="cuda")
    pf, pl = torch.from_numpy(s["prefix"]).cuda(), torch.from_numpy(s["plen"]).cuda()
    c = _lib.constraints(banned=s["banned"], **CON)
    ref = eng.beam_search(None, to_host=False, return_logprobs=True, beam_groups=2, diversity=0.3, length_penalty=0.5,
                          banned=s["banned"], **CON, **_pfx(s))
    assert eng.lib.fpnmt_beam_search_constrained_dl(eng._h, None, dl(pf), dl(pl), 2, C.c_float(0.3), C.c_float(0.5), C.byref(c),
                                                    dl(ids), dl(lens), dl(lp), 1, stream) == 0
    torch.cuda.synchronize()
    assert torch.equal(ids, ref[0]) and torch.equal(lens, ref[1]) and torch.equal(lp, ref[2])
    sp = _lib.sampling(**SAMPLING)
    ref = eng.sample(None, to_host=False, return_logprobs=True, banned=s["banned"], **CON, **SAMPLING)
    assert eng.lib.fpnmt_sample_constrained_dl(eng._h, None, None, None, C.byref(sp), C.byref(c), dl(ids), dl(lens), dl(lp), 1,
                                               stream) == 0
    torch.cuda.synchronize()
    assert torch.equal(ids, ref[0]) and torch.equal(lens, ref[1]) and torch.equal(lp, ref[2])
    eng.close()
    # Pipeline: banned_words resolved through the tokenizer; unknown words and <end> refused
    from fpnmt.dataset import Tokenizer
    from fpnmt.pipeline import Pipeline
    w = O.caption_weights(BB, vocab=512, layers=6, seed=0, end_bias=END_BIAS)
    img = O.test_images(2, 512, seed=41)
    tok = Tokenizer.synthetic(512)
    pipe = Pipeline(None, None, 12, tokenizer=tok, weights=w, beam=4, precision="bf16")
    words = [k for k, v in sorted(tok.word_index.items(), key=lambda kv: kv[1]) if v >= 4][:3] + ["<start>"]
    wid = [tok.word_index[x] for x in words]
    out = pipe.beam_search_batch(img, 12, num_beams=6, length_penalty=0.8, return_logprobs=True, no_repeat_ngram=2, min_len=3,
                                 banned_words=words)
    ref = pipe.transformer.engine(2, 6, 12).beam_search(img, length_penalty=0.8, return_logprobs=True, no_repeat_ngram=2,
                                                        min_len=3, banned=wid)
    for a, b in zip(out, ref):
        assert np.array_equal(a, b.numpy())
    assert not np.isin(out[0], wid).any() and (out[1] >= 3).all()
    plain = pipe.sample_batch(img, 12, seed=1)
    assert all(np.array_equal(a, b) for a, b in zip(plain, pipe.sample_batch(img, 12, seed=1, banned_words=None)))
    for bad in (["<end>"], ["no-such-word-here"]):
        with pytest.raises(ValueError):
            pipe.beam_search_batch(img, 12, banned_words=bad)
        with pytest.raises(ValueError):
            pipe.sample_batch(img, 12, banned_words=bad)


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


def _bits(ban):
    """boolean (R, F) -> int32 words (R, ceil(F / 32))"""
    R, F = ban.shape
    pad = np.zeros((R, (F + 31) // 32 * 32), np.uint64)
    pad[:, :F] = ban
    words = (pad.reshape(R, -1, 32) << np.arange(32, dtype=np.uint64)).sum(-1)
    return words.astype(np.uint32).view(np.int32)


@pytest.mark.parametrize("R,K,F,exact", [(256, 512, 1000, True), (130, 256, 904, False), (77, 512, 8 * 129, True)])
def test_vocab_stats_mask_operator(R, K, F, exact):
    from fpnmt.engine import vocab_stats, vocab_stats_mask, vocab_stats_target
    x, w, bias = _op_case(R, K, F, exact, R + F)
    rng = np.random.default_rng(F)
    z64 = _bf16(x) @ _bf16(w) + bias.astype(np.float64)[None, :]
    ban = rng.random((R, F)) < 0.3
    ft = (F + 127) // 128
    zt = np.pad(z64, ((0, 0), (0, ft * 128 - F)), constant_values=-np.inf).reshape(R, ft, 128)
    top = np.argsort(-zt, axis=-1, kind="stable")[:, :, 0]
    ban[np.arange(R), top[:, 0]] = True                           # every row's first-tile maximum is banned
    ban[::3, :] |= (np.arange(F) // 128 == 1)[None, :]            # tile 1 of every third row entirely banned
    tgt = rng.integers(0, F, size=R).astype(np.int32)
    xd = torch.from_numpy(x).cuda()
    st0, va0, ix0 = vocab_stats(xd, w, bias)
    st, va, ix, tl = vocab_stats_mask(xd, w, torch.from_numpy(_bits(ban)), bias, target=tgt)
    st1, va1, ix1, tl1 = vocab_stats_mask(xd, w, torch.zeros((R, (F + 31) // 32), dtype=torch.int32), bias)
    _, _, _, tl0 = vocab_stats_target(xd, w, tgt, bias)
    torch.cuda.synchronize()
    assert torch.equal(st0.view(torch.int32), st.view(torch.int32))            # statistics stay unmasked
    for a, b in ((st0, st1), (va0, va1), (ix0, ix1)):                          # all-zero mask: fpnmt_op_vocab_stats
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    assert tl1 is None and torch.equal(tl0.view(torch.int32), tl.view(torch.int32))
    va, ix = va.cpu().numpy(), ix.cpu().numpy()
    banp = np.pad(ban, ((0, 0), (0, ft * 128 - F)), constant_values=True).reshape(R, ft, 128)
    zm = np.where(banp, -np.inf, zt)
    order = np.argsort(-zm, axis=-1, kind="stable")[:, :, :8]
    allowed = np.take_along_axis(~banp, order, -1)
    ref_idx = np.where(allowed, order + (np.arange(ft) * 128)[None, :, None], 0x7fffffff)
    ref_val = np.where(allowed, np.take_along_axis(zm, order, -1), -np.inf)
    assert (ix == 0x7fffffff).sum() >= (R // 3) * 8                            # the fully banned tiles are empty
    for r in range(R):
        for t in range(ft):
            ok = ix[r, t] != 0x7fffffff
            assert not ban[r, ix[r, t][ok]].any(), (r, t)
    if exact:
        assert np.array_equal(ix, ref_idx) and np.array_equal(va.astype(np.float64), ref_val)
    else:
        absprod = np.abs(_bf16(x)) @ np.abs(_bf16(w))
        delta = (K * 2.0 ** -23 * absprod.max(-1) + 2.0 ** -24 * np.abs(z64).max(-1))[:, None, None]
        ok = ref_idx != 0x7fffffff
        assert np.array_equal(ok, ix != 0x7fffffff)
        assert (np.abs(va[ok] - ref_val[ok]) <= np.broadcast_to(delta, ok.shape)[ok]).all()
        with np.errstate(invalid="ignore"):                                       # -inf - -inf in short tiles
            gaps = np.diff(np.sort(zm, -1)[:, :, ::-1][:, :, :9], axis=-1)
        clear = (np.abs(gaps) > 2 * delta).all(-1)                                 # no near-tie among the top 9
        assert clear.mean() > 0.5
        assert (np.sort(ix, -1) == np.sort(ref_idx, -1))[clear].all()


def test_ban_mask_operator():
    from fpnmt.engine import ban_mask
    rng = np.random.default_rng(9)
    R, LD, Vs, end = 300, 16, 100, 3
    hist = rng.integers(0, 6, size=(R, LD)).astype(np.int32)     # six ids: many repeated n-grams
    hist[::5] = rng.integers(0, Vs, size=(R // 5, LD))
    lens = rng.integers(0, LD + 1, size=R).astype(np.int32)
    lens[0], lens[1] = -2, LD + 5                                  # clamped to [0, ld]
    for n, min_len, banned in ((0, 0, None), (1, 4, [7, 99]), (2, 0, [0]), (3, 9, [5, 5, 64]), (4, LD, None)):
        got = ban_mask(hist, lens, Vs, end, n, min_len, banned).cpu().numpy()
        ref = np.stack([CO.ban_set(hist[r, :min(max(lens[r], 0), LD)], Vs, end, n, min_len, banned) for r in range(R)])
        assert np.array_equal(got, _bits(ref)), (n, min_len, banned)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_ban_masks_live_on_the_engines_gpu_when_another_gpu_is_current(subject):
    # engine A's first constrained call comes after another engine made GPU 1 the thread's current device
    s = subject
    a = _engine(s, device=0)
    _load_memory(a, s)
    _search(a, **_pfx(s, length_penalty=0.8))
    b = _engine(s, device=1)
    b.generate(s["img"], early_stop=False)
    torch.cuda.set_device(1)
    got = _search(a, **_pfx(s, length_penalty=0.8), **CON, banned=s["banned"])
    torch.cuda.set_device(0)
    b.close()
    ref = _search(a, **_pfx(s, length_penalty=0.8), **CON, banned=s["banned"])
    a.close()
    for x, y in zip(got, ref):
        assert np.array_equal(x, y)
    _check(s, got[0], got[1], CON, s["banned"], s["plen"])
