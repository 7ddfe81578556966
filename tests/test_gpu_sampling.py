"""Sampled caption decoding (Engine.sample / fpnmt_sample, fpnmt_op_sample_step) against the fp64 oracle of
tests/sample_oracle.py.

Bounds.
  operator token   equal on every row whose margin (sample_oracle.sample_step: distance of u * mass from a CDF step, and of
                   the nucleus target from a cumulative mass at which K2 changes, as a fraction of the mass) exceeds 1e-6.  The
                   kernel's probabilities are fp32 expf of fp32 (z - max) / temperature (a few ulp, ~5e-7 relative), held as
                   integers at 2^-40 of the row maximum's probability (at most V * 2^-41 / 1 <= 2.3e-8 of the mass for
                   V <= 51200); both are below 1e-6.  The top-k decision compares the same fp32 logits exactly.
  operator u       bit-equal: (philox[0] >> 8) * 2^-24 is exact in fp32 and fp64.
  operator logprob 1e-5: z[token] - max - log(sum exp(z - max)), fp32 sum of V <= 10 000 terms with relative error
                   <= ~1e-6 in practice, log of it absolute.
  end to end       bf16x3 holds teacher-forced log-probabilities within 2e-3 per step (tests/test_gpu_captions.py), so a
                   caption's log-likelihood over len + 1 steps within 2e-3 * (len + 1); a draw whose u lies within that
                   perturbation of a CDF step may differ from the oracle's, after which the sample diverges: >= 95 % of the
                   samples are required to be identical.
  bf16 greedy      exact: the sampler's temperature-0 path and the reference beam search with identical beams pick the same
                   arg-max of the same logits (same layer kernels, same fp32 emb + pos input) unless two logits tie exactly.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import fpnmt_oracle as O
import sample_oracle as SO

pytestmark = pytest.mark.gpu

BB, S, L, V, T, N, B = "mobilenet224_1.0", 256, 2, 512, 16, 8, 8


def _rows(V, rows, kind, seed):
    rng = np.random.default_rng(seed)
    z = (rng.normal(size=(rows, V)) * 2.5).astype(np.float32)
    for r in range(rows):
        c = (r + kind) % 5
        if c == 1:                                            # a second arg-max
            z[r, rng.integers(V)] = z[r].max()
        elif c == 2:                                          # ties at the 5-th largest logit
            v = np.sort(z[r])[::-1][4]
            z[r, rng.choice(V, 3, replace=False)] = v
        elif c == 3:                                          # Pipeline's padded vocabulary entries
            z[r, V - V // 8:] = -1e9
        elif c == 4:                                          # coarse logits: many exact ties in p (nucleus boundary)
            z[r] = np.round(z[r] * 2) / 2
    return z


OP_CASES = [(v, tp, k, p) for v in (512, 1000, 10000) for tp in (0.0, 0.5, 1.0, 1.7) for k in (0, 1, 5, "V")
            for p in (1.0, 0.9, 0.3, 1e-6)]


@pytest.mark.parametrize("V_", [512, 1000, 10000])
def test_operator_matches_fp64_oracle(V_):
    from fpnmt.engine import sample_step
    rows, spi = 40, 8
    excluded = total = 0
    worst_lp = 0.0
    for ci, (v, temp, k, p) in enumerate(c for c in OP_CASES if c[0] == V_):
        k = V_ if k == "V" else k
        z = _rows(V_, rows, ci, seed=1000 + ci)
        t, seed = ci % 7, 0x123456789 + ci
        tok, lp, u = (x.cpu().numpy() for x in sample_step(torch.from_numpy(z).cuda(), spi, t, temp, k, p, seed))
        params = dict(temperature=temp, top_k=k, top_p=p, seed=seed)
        for r in range(rows):
            ref = SO.sample_step(z[r], r // spi, r % spi, t, params)
            assert float(u[r]) == ref["u"], (v, temp, k, p, r)
            total += 1
            if ref["margin"] <= 1e-6:
                excluded += 1
                continue
            assert ref["K2"][tok[r]], ("token outside K2", v, temp, k, p, r)
            assert tok[r] == ref["token"], (v, temp, k, p, r, tok[r], ref["token"], ref["margin"])
            worst_lp = max(worst_lp, abs(float(lp[r]) - ref["logprob"]))
    print("V=%d: %d rows, %d excluded at a boundary, worst log-prob error %.2e" % (V_, total, excluded, worst_lp))
    assert worst_lp <= 1e-5
    assert excluded <= total // 100


# seeds whose uniform at counter (0, 0, 0, 0) is exactly 1/2, 3/4 and 1/4 (found by search over the oracle's Philox)
EXACT_U = [(515707, 0.5), (22356995, 0.75), (23739184, 0.25)]


def test_draw_is_strictly_above_u_on_exact_cdf_steps():
    """Four equal logits: the cumulative mass steps are exact quarters, and so are these u.  The token is the first whose
    cumulative mass is strictly greater than u * mass: 1 + 4u, not 4u."""
    from fpnmt.engine import sample_step
    z = torch.tensor([[0.0] * 4 + [-1e9] * 4])
    for seed, uu in EXACT_U:
        tok, _, u = sample_step(z.cuda(), 1, 0, 1.0, 0, 1.0, seed)
        ref = SO.sample_step(z[0].numpy(), 0, 0, 0, dict(seed=seed))
        assert float(u[0]) == uu == ref["u"]
        assert int(tok[0]) == ref["token"] == int(4 * uu), (seed, int(tok[0]))


def test_draws_follow_the_truncated_distribution():
    from scipy.stats import chisquare
    from fpnmt.engine import sample_step
    rows, Vd = 16384, 64
    z = (np.random.default_rng(7).normal(size=Vd) * 1.5).astype(np.float32)
    params = dict(temperature=0.8, top_k=20, top_p=0.95, seed=99)
    tok, _, _ = sample_step(torch.from_numpy(np.tile(z, (rows, 1))).cuda(), 16, 3, **params)
    tok = tok.cpu().numpy()
    ref = SO.sample_step(z, 0, 0, 3, params)
    K2, q = ref["K2"], ref["q"]
    assert K2[tok].all(), "a draw outside K2"
    assert 5 <= K2.sum() < 20                                 # both filters bite on this row
    counts = np.bincount(tok, minlength=Vd)[K2]
    stat, pval = chisquare(counts, q[K2] * rows)
    print("chi-square %.1f over %d tokens, p = %.3g" % (stat, K2.sum(), pval))
    assert pval > 1e-4


@pytest.fixture(scope="module")
def subject():
    w = O.caption_weights(BB, vocab=V, layers=L, seed=0, end_bias=6.0)
    Wv = O.W(w)
    img = O.test_images(B, S, seed=41)
    with torch.no_grad():
        mem = O.encoder(img, Wv, BB, num_layers=L, input_vocab_size=(S // 16) ** 2)
    g_ids, g_len = O.predict_batch_cached(mem, Wv, T, N, 2, 3, num_layers=L)
    return dict(w=w, Wv=Wv, img=img, mem=mem, g_ids=g_ids, g_len=g_len)


def _engine(s, prec="bf16", **kw):
    from fpnmt.engine import Engine
    return Engine(s["w"], backbone=BB, batch=B, beam=N, vocab=V, max_len=T, num_layers=L, image_size=S, precision=prec, **kw)


def _load_memory(eng, s):
    eng.decode_logits(s["mem"].cuda(), torch.full((B, 1), 2, dtype=torch.int32).cuda())


@pytest.mark.parametrize("temp,k,p", [(1.0, 0, 0.9), (0.7, 10, 1.0)])
def test_end_to_end_bf16x3_matches_oracle(subject, temp, k, p):
    s = subject
    ref_ids, ref_len, ref_lp = SO.sample_batch_cached(s["mem"], s["Wv"], T, N, 2, 3, temperature=temp, top_k=k, top_p=p, seed=7,
                                                      num_layers=L)
    # the subject is not degenerate: samples leave the greedy caption, differ per image, and end mid-sequence
    greedy = (ref_ids == s["g_ids"][:, None]).all(-1) & (ref_len == s["g_len"][:, None])
    assert greedy.mean() < 0.5
    assert np.mean([len({tuple(ref_ids[b, n, :ref_len[b, n]]) for n in range(N)}) for b in range(B)]) >= 3
    assert ((ref_len > 0) & (ref_len < T)).sum() >= 8
    eng = _engine(s, "bf16x3")
    _load_memory(eng, s)
    ids, lens, lp = eng.sample(None, temperature=temp, top_k=k, top_p=p, seed=7, return_logprobs=True)
    eng.close()
    ids, lens, lp = ids.numpy(), lens.numpy(), lp.numpy()
    same = (ids == ref_ids).all(-1) & (lens == ref_len)
    print("(%g, %d, %g): %d / %d samples identical" % (temp, k, p, same.sum(), same.size))
    assert same.mean() >= 0.95
    err = np.abs(lp - ref_lp)[same] / (lens[same] + 1)
    assert float(err.max()) <= 2e-3, float(err.max())
    assert ((ids != 0).sum(-1) <= lens).all()                 # nothing written after a sample finished


def test_bf16_greedy_equals_generate(subject):
    s = subject
    trace = {}
    SO.sample_batch_cached(s["mem"], s["Wv"], T, 1, 2, 3, temperature=0.0, num_layers=L, trace=trace)
    assert min(trace["top2_gap"]) > 0.0                       # no exact top-1 tie on the greedy path
    eng = _engine(s, opts=("no_vstats",))
    g_ids, g_len = eng.generate(s["img"], early_stop=True)
    ids, lens = eng.sample(None, temperature=0.0, seed=3)
    eng.close()
    for n in range(N):
        assert torch.equal(ids[:, n], g_ids) and torch.equal(lens[:, n], g_len), n


def _run(eng, **kw):
    return [x.clone() for x in eng.sample(None, return_logprobs=True, **kw)]


def test_bf16_bit_identical_across_graphs_early_stop_and_cache_modes(subject):
    s = subject
    kw = dict(temperature=0.9, top_k=20, top_p=0.95, seed=11)
    outs = []
    for opts in (dict(use_graphs=True), dict(use_graphs=False), dict(use_graphs=True, cache_mode="physical")):
        eng = _engine(s, **opts)
        _load_memory(eng, s)
        for es in (True, False):
            outs.append(_run(eng, early_stop=es, **kw))
        outs.append(_run(eng, early_stop=True, **kw))                  # same seed again: same bits
        other = _run(eng, early_stop=True, **dict(kw, seed=12))
        eng.close()
        differ = ~((other[0] == outs[-1][0]).all(-1) & (other[1] == outs[-1][1]))
        assert differ.float().mean() >= 0.5, differ.float().mean()    # another seed changes most samples
    for o in outs[1:]:
        for a, b in zip(o, outs[0]):
            assert torch.equal(a, b)
    assert ((outs[0][1] > 0) & (outs[0][1] < T)).any()


def test_sampling_leaves_generate_unchanged(subject):
    s = subject
    for cache_mode in ("ancestry", "physical"):
        eng = _engine(s, cache_mode=cache_mode)
        a = eng.generate(s["img"], early_stop=False)
        eng.sample(None, temperature=1.3, top_k=0, top_p=1.0, seed=5)
        eng.sample(s["img"], temperature=0.5, top_k=3, top_p=0.5, seed=6, early_stop=False)
        b = eng.generate(s["img"], early_stop=False)
        eng.close()
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_errors_launch_count_and_dlpack(subject):
    from fpnmt import _lib
    from fpnmt._lib import FpnmtError
    s = subject
    fused = _engine(s, decode_path="fused")
    with pytest.raises(FpnmtError) as ei:
        fused.sample(s["img"])
    assert ei.value.code == _lib.ERR_STATE
    fused.close()
    eng = _engine(s)
    _load_memory(eng, s)
    for bad in (dict(temperature=-0.1), dict(top_p=0.0), dict(top_p=1.5), dict(top_k=-1), dict(top_k=V + 1)):
        with pytest.raises(FpnmtError) as ei:
            eng.sample(None, **bad)
        assert ei.value.code == _lib.ERR_INVALID, bad
    stream = torch.cuda.current_stream().cuda_stream
    ids = torch.zeros((B, N, T), dtype=torch.int32, device="cuda")
    lens = torch.zeros((B, N), dtype=torch.int32, device="cuda")
    sp = _lib.sampling(1.0, 0, 1.0, 1)
    sp.reserved[2] = 1
    assert eng.lib.fpnmt_sample(eng._h, None, 0, C.byref(sp), ids.data_ptr(), lens.data_ptr(), None, 0, 1, stream) == _lib.ERR_INVALID
    assert eng.lib.fpnmt_sample(eng._h, None, 0, None, ids.data_ptr(), lens.data_ptr(), None, 0, 1, stream) == _lib.ERR_INVALID
    # launch count: per step the teacher-forced program + 1 (decode_logits: + 2), plus k_sample_init once
    tok = torch.full((B, T), 2, dtype=torch.int32).cuda()
    c0 = eng.launch_count
    eng.decode_logits(s["mem"].cuda(), tok)
    c1 = eng.launch_count
    eng.sample(None, early_stop=False, seed=4)
    c2 = eng.launch_count
    assert (c2 - c1) - (c1 - c0) == 1 - T
    # DLPack twin == raw entry point
    ref = eng.sample(None, temperature=0.8, top_k=7, seed=21, to_host=False, return_logprobs=True)
    lp = torch.zeros((B, N), dtype=torch.float32, device="cuda")
    keep = []

    def dl(x):
        p, k = _lib.dl_tensor(x)
        keep.append(k)
        return p
    sp = _lib.sampling(0.8, 7, 1.0, 21)
    assert eng.lib.fpnmt_sample_dl(eng._h, None, C.byref(sp), dl(ids), dl(lens), dl(lp), 1, stream) == 0
    torch.cuda.synchronize()
    assert torch.equal(ids, ref[0]) and torch.equal(lens, ref[1]) and torch.equal(lp, ref[2])
    bad_ids = torch.zeros((B, N, T + 1), dtype=torch.int32, device="cuda")
    assert eng.lib.fpnmt_sample_dl(eng._h, None, C.byref(sp), dl(bad_ids), dl(lens), None, 1, stream) == _lib.ERR_INVALID
    eng.close()
    # lane 0 holding a submitted batch
    lanes = _engine(s, lanes=2)
    keep_img = lanes.submit(0, s["img"].cuda(), early_stop=False)
    with pytest.raises(FpnmtError) as ei:
        lanes.sample(None)
    assert ei.value.code == _lib.ERR_STATE
    lanes.collect(0)
    del keep_img
    lanes.close()


def test_pipeline_sample_batch():
    from fpnmt.dataset import Tokenizer
    from fpnmt.pipeline import Pipeline
    w = O.caption_weights(BB, vocab=V, layers=6, seed=0, end_bias=56.0)
    img = O.test_images(2, 512, seed=41)
    pipe = Pipeline(None, None, 12, tokenizer=Tokenizer.synthetic(V), weights=w, beam=4, precision="bf16")
    g_ids, g_len = pipe.predict_batch(img, 12)
    ids, lens, lp = pipe.sample_batch(img, 12, temperature=0.0, return_logprobs=True)
    assert ids.shape == (2, 4, 12) and lens.shape == (2, 4) and lp.shape == (2, 4) and (lp < 0).all()
    for n in range(4):
        assert (ids[:, n] == g_ids).all() and (lens[:, n] == g_len).all()
    ids6, lens6 = pipe.sample_batch(img, 12, num_samples=6, temperature=1.0, top_p=0.9, seed=1)
    assert ids6.shape == (2, 6, 12) and lens6.shape == (2, 6)
