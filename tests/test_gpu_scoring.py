"""Caption scoring (Engine.score / fpnmt_score, Pipeline.score_batch) against the fp64 oracle and the engine's own slow path.

Reference.  fpnmt_oracle.decode.teacher_forced_logprobs on [<start>] + caption with fp64 weights (O.W(w, torch.float64)),
fed the memory the engine holds; the term of position j is its log-probability of ids[j] for j < len and of <end> at
j = len < t.  Captions are random ids in [4, V) with lengths mixed within an image, including len = 0 (only <end>) and
len = t (no <end>).

Bounds (absolute).
  bf16x3  2e-3 per term and 2e-3 * n_bn per caption: the project's teacher-forced bound for this mode
          (tests/test_gpu_captions.py, test_gpu_engine.py).
  bf16    0.25 per caption and scored position (|total error| / n_bn): the bf16 decoder bound of tests/test_gpu_engine.py
          at logit std ~6 (this subject: 6.1).  Per term 0.5: that bound is the worst of 64 terms, one caption per image;
          here up to 960 terms per case are compared, and the worst term of the existing KV-cached path (decode_logits)
          against the same oracle, printed by test_bf16_matches_the_slow_path, is of the same size as the score pass's
          (NVIDIA B200: 0.29 .. 0.33 for the score pass over these cases).  That test also holds the score pass to the
          existing path's own worst error plus the pass-to-pass bound below.
  bf16    0.2 per term against this engine's own slow path (decode_logits, `no_xattn`: the same cross-attention kernel;
          log_softmax and gather in torch).  Both passes round every activation to bf16 at the same points and accumulate in
          fp32; they differ only in the order of the fp32 sums (tgemm at B * N rows vs igemm at B * N * t rows, a KV cache vs
          the QKV projection in the self-attention).  An activation therefore differs by at most one bf16 ulp (2^-8
          relative) where the two sums straddle a rounding boundary, and the terms move by a fraction of either pass's error
          against fp64: measured worst 0.13 (NVIDIA B200, 1000 W), the bound 1.5x that.
  sampling  on bf16x3 score(sample(...)) = the sample's out_logprob within 2e-3 * (len + 1): both are the same caption's
          terms from two bf16x3 passes, each within 2e-3 per term of the oracle's.
Kernel mutations (causal off by one, position off by one, swapped heads, dropped <end> term, cross-attention image index
with N instead of N * t, caption sum past n_bn, no online-softmax rescale at a chunk boundary) each fail
test_matches_fp64_oracle.
Exact properties (bit-equal): run to run, graphs on / off, captions permuted within an image, ids at positions >= len
overwritten, and the other captions of a batch in which one caption is invalid.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import fpnmt_oracle as O

pytestmark = pytest.mark.gpu

BB, L, V, B = "mobilenet224_1.0", 2, 512, 4
TOL = {"bf16x3": 2e-3, "bf16": 0.5}           # per term
TOL_TOT = {"bf16x3": 2e-3, "bf16": 0.25}      # per caption, divided by n_bn
TOL_SLOW = 0.2
# (image size S -> 4 or 16 memory tokens, captions per image N, positions t, engine max_len, cache_mode)
CASES = [(256, 1, 1, 16, "ancestry"), (256, 3, 16, 16, "physical"), (512, 8, 16, 16, "ancestry"), (512, 3, 9, 16, "physical"),
         (256, 3, 80, 80, "ancestry")]
_SUBJECTS = {}


def subject(S):
    if S not in _SUBJECTS:
        w = O.caption_weights(BB, vocab=V, layers=L, seed=0, end_bias=6.0)
        img = O.test_images(B, S, seed=41)
        with torch.no_grad():
            mem = O.encoder(img, O.W(w), BB, num_layers=L, input_vocab_size=(S // 16) ** 2).to(torch.float32)
        _SUBJECTS[S] = dict(w=w, W64=O.W(w, torch.float64), img=img, mem=mem)
    return _SUBJECTS[S]


def captions(N, t, seed):
    """ids (B, N, t) int32 in [4, V), lens (B, N): random, with len 0 and len t present and mixed lengths in an image."""
    rng = np.random.default_rng(seed)
    ids = rng.integers(4, V, size=(B, N, t)).astype(np.int32)
    lens = rng.integers(0, t + 1, size=(B, N)).astype(np.int32)
    lens[0, 0], lens[1, N - 1] = 0, t
    if t > 1:
        lens[2, 0] = t - 1
    return ids, lens


def oracle(s, ids, lens):
    """fp64 teacher-forced terms (B, N, t) (0 past n_bn) and totals (B, N)."""
    Bn, N, t = ids.shape
    tok = np.full((Bn, N, t), 2, np.int64)
    tok[:, :, 1:] = ids[:, :, :t - 1]
    tgt = ids.astype(np.int64).copy()
    mask = np.zeros((Bn, N, t), bool)
    for b in range(Bn):
        for n in range(N):
            ln = int(lens[b, n])
            if ln < t:
                tgt[b, n, ln] = 3
            mask[b, n, :min(ln + 1, t)] = True
    mem = s["mem"].double().repeat_interleave(N, 0)
    with torch.no_grad():
        lp = O.teacher_forced_logprobs(mem, torch.from_numpy(tok.reshape(-1, t)), s["W64"], t, L).double().numpy()
    terms = np.take_along_axis(lp.reshape(Bn, N, t, -1), tgt[..., None], -1)[..., 0] * mask
    return terms, terms.sum(-1)


def _engine(s, S, N, T, prec="bf16", **kw):
    from fpnmt.engine import Engine
    return Engine(s["w"], backbone=BB, batch=B, beam=N, vocab=V, max_len=T, num_layers=L, image_size=S, precision=prec, **kw)


def _load_memory(eng, s):
    eng.decode_logits(s["mem"].cuda(), torch.full((B, 1), 2, dtype=torch.int32).cuda())


def _score(eng, ids, lens, images=None):
    lp, tl = eng.score(torch.from_numpy(ids).cuda(), torch.from_numpy(lens).cuda(), images, return_token_logprobs=True)
    return lp.numpy().astype(np.float64), tl.numpy().astype(np.float64)


def _n_bn(lens, t):
    return np.where(lens < t, lens + 1, t)


@pytest.mark.parametrize("prec", ["bf16x3", "bf16"])
@pytest.mark.parametrize("S,N,t,T,cache_mode", CASES)
def test_matches_fp64_oracle(prec, S, N, t, T, cache_mode):
    s = subject(S)
    ids, lens = captions(N, t, seed=S + 10 * N + t)
    ref_terms, ref_tot = oracle(s, ids, lens)
    assert ref_terms.std() > 1.0                                       # the terms are not flat
    eng = _engine(s, S, N, T, prec, cache_mode=cache_mode)
    _load_memory(eng, s)
    lp, tl = _score(eng, ids, lens)
    eng.close()
    n_bn = _n_bn(lens, t)
    beyond = np.arange(t)[None, None, :] >= n_bn[..., None]
    assert (tl[beyond] == 0).all()
    err = np.abs(tl - ref_terms).max()
    err_tot = (np.abs(lp - ref_tot) / n_bn).max()
    print("%s S=%d N=%d t=%d: worst term error %.2e (%.3f of the bound), worst total error / n_bn %.2e"
          % (prec, S, N, t, err, err / TOL[prec], err_tot))
    assert err <= TOL[prec]
    assert err_tot <= TOL_TOT[prec]
    # the sum is the position-ordered sum of the terms (fp32 on the device)
    np.testing.assert_allclose(lp, tl.sum(-1), rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("S,N,t,T,cache_mode", CASES)
def test_bf16_matches_the_slow_path(S, N, t, T, cache_mode):
    """The same numbers the slow way: N teacher-forced decode_logits calls (KV-cached step program, `no_xattn` so the
    cross-attention kernel is the one the score pass uses), log_softmax and gather in torch."""
    s = subject(S)
    ids, lens = captions(N, t, seed=S + 10 * N + t)
    ref_terms, _ = oracle(s, ids, lens)
    eng = _engine(s, S, N, T, "bf16", cache_mode=cache_mode, opts=("no_xattn",))
    _load_memory(eng, s)
    lp, tl = _score(eng, ids, lens)
    slow = np.zeros((B, N, t))
    for n in range(N):
        tok = np.full((B, t), 2, np.int32)
        tok[:, 1:] = ids[:, n, :t - 1]
        lsm = torch.log_softmax(eng.decode_logits(s["mem"].cuda(), torch.from_numpy(tok).cuda()), -1).double().cpu().numpy()
        for b in range(B):
            ln = int(lens[b, n])
            tgt = list(ids[b, n, :ln]) + ([3] if ln < t else [])
            slow[b, n, :len(tgt)] = lsm[b, np.arange(len(tgt)), tgt]
    eng.close()
    err = np.abs(tl - slow).max()
    slow_err, score_err = np.abs(slow - ref_terms).max(), np.abs(tl - ref_terms).max()
    print("bf16 vs slow path S=%d N=%d t=%d: worst term difference %.2e; worst term error against fp64: slow path %.2e, "
          "score %.2e" % (S, N, t, err, slow_err, score_err))
    assert err <= TOL_SLOW
    assert score_err <= slow_err + TOL_SLOW
    assert (np.abs(lp - slow.sum(-1)) / _n_bn(lens, t)).max() <= TOL_SLOW


def test_bf16x3_score_of_samples_equals_their_logprob():
    S, N, T = 256, 8, 16
    s = subject(S)
    eng = _engine(s, S, N, T, "bf16x3")
    _load_memory(eng, s)
    ids, lens, lp = eng.sample(None, temperature=1.0, top_k=0, top_p=0.9, seed=7, return_logprobs=True)
    ids, lens, lp = ids.numpy(), lens.numpy(), lp.numpy().astype(np.float64)
    # the subject is not degenerate: samples end mid-sequence, some run T steps, and they differ within an image
    assert ((lens > 0) & (lens < T)).sum() >= 3 and (lens == T).any()
    assert np.mean([len({tuple(ids[b, n, :lens[b, n]]) for n in range(N)}) for b in range(B)]) >= 3
    sc = eng.score(torch.from_numpy(ids).cuda(), torch.from_numpy(lens).cuda()).numpy().astype(np.float64)
    eng.close()
    err = (np.abs(sc - lp) / (lens + 1)).max()
    print("score(sample) vs the sample's log-prob: worst error / (len + 1) %.2e" % err)
    assert err <= 2e-3


def test_bit_identical_graphs_permutation_and_ignored_positions():
    S, N, t, T = 256, 3, 80, 80
    s = subject(S)
    ids, lens = captions(N, t, seed=5)
    outs = []
    for graphs in (True, False):
        eng = _engine(s, S, N, T, "bf16", use_graphs=graphs)
        _load_memory(eng, s)
        outs += [_score(eng, ids, lens), _score(eng, ids, lens)]
        if graphs:
            perm = np.array([2, 0, 1])
            pl, pt = _score(eng, ids[:, perm], lens[:, perm])
            assert np.array_equal(pl, outs[0][0][:, perm]) and np.array_equal(pt, outs[0][1][:, perm])
            junk = ids.copy()
            rng = np.random.default_rng(9)
            for b in range(B):
                for n in range(N):
                    junk[b, n, lens[b, n]:] = rng.integers(0, V, size=t - lens[b, n])
            jl, jt = _score(eng, junk, lens)
            assert np.array_equal(jl, outs[0][0]) and np.array_equal(jt, outs[0][1])
        eng.close()
    for o in outs[1:]:
        assert np.array_equal(o[0], outs[0][0]) and np.array_equal(o[1], outs[0][1])


def test_invalid_captions_are_nan_and_leave_the_others_alone():
    S, N, t, T = 256, 3, 16, 16
    s = subject(S)
    ids, lens = captions(N, t, seed=6)
    lens[:, :] = np.maximum(lens, 3)
    lens[3, 0] = 5
    eng = _engine(s, S, N, T, "bf16")
    _load_memory(eng, s)
    clean_l, clean_t = _score(eng, ids, lens)
    bad_ids, bad_lens = ids.copy(), lens.copy()
    bad_lens[0, 1] = -1
    bad_lens[1, 0] = t + 1
    bad_ids[2, 2, 1] = V                 # ids just past the vocabulary, inside the caption
    bad_ids[3, 1, lens[3, 1] - 1] = V + 7
    bad_ids[3, 0, lens[3, 0]] = V + 7    # past the caption: ignored
    lp, tl = _score(eng, bad_ids, bad_lens)
    eng.close()
    bad = np.zeros((B, N), bool)
    bad[0, 1] = bad[1, 0] = bad[2, 2] = bad[3, 1] = True
    assert np.isnan(lp[bad]).all() and np.isnan(tl[bad]).all()
    assert np.array_equal(lp[~bad], clean_l[~bad]) and np.array_equal(tl[~bad], clean_t[~bad])


def test_scoring_leaves_generate_sample_and_launch_count_unchanged():
    S, N, T = 256, 3, 16
    s = subject(S)
    ids, lens = captions(N, 16, seed=7)
    for cache_mode in ("ancestry", "physical"):
        eng = _engine(s, S, N, T, "bf16", cache_mode=cache_mode)
        g0 = eng.generate(s["img"], early_stop=False)
        s0 = eng.sample(None, temperature=0.9, top_p=0.9, seed=3, return_logprobs=True)
        _score(eng, ids, lens)
        _score(eng, ids[:, :, :7], np.minimum(lens, 7), s["img"])
        g1 = eng.generate(s["img"], early_stop=False)
        s1 = eng.sample(None, temperature=0.9, top_p=0.9, seed=3, return_logprobs=True)
        for a, b in zip(g0 + s0, g1 + s1):
            assert torch.equal(a, b), cache_mode
        counts = []
        for _ in range(3):
            c = eng.launch_count
            _score(eng, ids, lens)
            counts.append(eng.launch_count - c)
        assert counts[0] == counts[1] == counts[2] > 0, counts
        eng.close()


def test_errors_dlpack_and_pipeline():
    from fpnmt import _lib
    from fpnmt._lib import FpnmtError
    S, N, t, T = 256, 3, 16, 16
    s = subject(S)
    ids, lens = captions(N, t, seed=8)
    dids, dlens = torch.from_numpy(ids).cuda(), torch.from_numpy(lens).cuda()
    fused = _engine(s, S, N, T, "bf16", decode_path="fused")
    with pytest.raises(FpnmtError) as ei:
        fused.score(dids, dlens, s["img"])
    assert ei.value.code == _lib.ERR_STATE
    fused.close()
    eng = _engine(s, S, N, T, "bf16")
    _load_memory(eng, s)
    stream = torch.cuda.current_stream().cuda_stream
    lp = torch.zeros((B, N), dtype=torch.float32, device="cuda")
    tl = torch.zeros((B, N, t), dtype=torch.float32, device="cuda")
    for bad_t in (0, T + 1):
        assert eng.lib.fpnmt_score(eng._h, None, 0, dids.data_ptr(), dlens.data_ptr(), bad_t, lp.data_ptr(), None, 0, stream) == _lib.ERR_INVALID
    for args in ((None, dlens.data_ptr(), lp.data_ptr()), (dids.data_ptr(), None, lp.data_ptr()), (dids.data_ptr(), dlens.data_ptr(), None)):
        assert eng.lib.fpnmt_score(eng._h, None, 0, args[0], args[1], t, args[2], None, 0, stream) == _lib.ERR_INVALID
    # DLPack twin == raw entry point
    ref_l, ref_t = eng.score(dids, dlens, to_host=False, return_token_logprobs=True)
    keep = []

    def dl(x):
        p, k = _lib.dl_tensor(x)
        keep.append(k)
        return p
    assert eng.lib.fpnmt_score_dl(eng._h, None, dl(dids), dl(dlens), dl(lp), dl(tl), stream) == 0
    torch.cuda.synchronize()
    assert torch.equal(lp, ref_l) and torch.equal(tl, ref_t)
    bad_tl = torch.zeros((B, N, t + 1), dtype=torch.float32, device="cuda")
    assert eng.lib.fpnmt_score_dl(eng._h, None, dl(dids), dl(dlens), dl(lp), dl(bad_tl), stream) == _lib.ERR_INVALID
    bad_lens = torch.zeros((B, N + 1), dtype=torch.int32, device="cuda")
    assert eng.lib.fpnmt_score_dl(eng._h, None, dl(dids), dl(bad_lens), dl(lp), None, stream) == _lib.ERR_INVALID
    eng.close()
    # lane 0 holding a submitted batch
    lanes = _engine(s, S, N, T, "bf16", lanes=2)
    keep_img = lanes.submit(0, s["img"].cuda(), early_stop=False)
    with pytest.raises(FpnmtError) as ei:
        lanes.score(dids, dlens)
    assert ei.value.code == _lib.ERR_STATE
    lanes.collect(0)
    del keep_img
    lanes.close()
    # Pipeline.score_batch: texts of the synthetic tokenizer -> the same bits as Engine.score on the tokenized ids
    from fpnmt.dataset import Tokenizer
    from fpnmt.pipeline import Pipeline
    w6 = O.caption_weights(BB, vocab=V, layers=6, seed=0, end_bias=6.0)
    img = O.test_images(2, 512, seed=41)
    pipe = Pipeline(None, None, 12, tokenizer=Tokenizer.synthetic(V), weights=w6, beam=4, precision="bf16")
    texts = [["<start> w5 w17 w100 <end>", "w9", "", "w4 w4 w4 w4 w4 w4 w4 w4 w4 w4 w4 w4"],
             ["w300 w301", "<start> w7 w8 w9 <end>", "w511 w6", "w44 w45 w46"]]
    got, got_t = pipe.score_batch(img, texts, return_token_logprobs=True)
    toks = [[[5, 17, 100], [9], [], [4] * 12], [[300, 301], [7, 8, 9], [511, 6], [44, 45, 46]]]
    t_p = 12
    pid = np.zeros((2, 4, t_p), np.int32)
    plen = np.zeros((2, 4), np.int32)
    for b in range(2):
        for n in range(4):
            pid[b, n, :len(toks[b][n])] = toks[b][n]
            plen[b, n] = len(toks[b][n])
    ref_l, ref_t = pipe.transformer.engine(2, 4, 12).score(pid, plen, img, return_token_logprobs=True)
    assert got.shape == (2, 4) and got_t.shape == (2, 4, t_p) and (got < 0).all()
    assert np.array_equal(got, ref_l.numpy()) and np.array_equal(got_t, ref_t.numpy())
    with pytest.raises(ValueError):
        pipe.score_batch(img, [["w5 " * 13] * 4, ["w5"] * 4])
