"""Decoder attention weights (Engine.decode_attention / caption_attention, fpnmt_decode_attention) against the fp64 oracle.

Test subject.  Under `test_weights` the cross-attention is nearly uniform (mean max-probability 0.33 over 4 tokens), so a
wrong head or token index could hide inside a bf16 bound.  Each layer's mha2/wq kernel is multiplied by 4 (mean
max-probability 0.54 over 4 tokens, 0.31 over 16; median max-abs difference between head h and head h+1: 0.26..0.45) and
its bias by 100 (std 2): the query bias then moves the cross-attention by >= 0.2, so the score-bias term of the fused
cross-attention block is visible too.  Self-attention is sharp already (0.30..0.46).  Every test asserts these properties
of its reference before it compares anything.

Bounds (max-abs over every probability).
  bf16x3  2e-3: softmax is 1-Lipschitz from log-probabilities, |dp| <= p |d log p| <= |d log p| for p <= 1, and this mode
          holds teacher-forced log-probabilities of the vocabulary softmax within 2e-3 (tests/test_gpu_captions.py); the
          attention scores come from the same fp32-class activations.
  bf16    5e-2: below a third of the smallest median head-swap difference (0.26), so a wrong head or token still fails;
          the fused cross-attention block keeps bf16 folded operands (tests/test_gpu_engine.py: 5e-2 relative on logits).
  captions (Pipeline.predict, bf16x3 end to end from the image, 6 layers) are held to the bf16x3 bound as well.
Measured worst values (NVIDIA B200, 1000 W power limit): bf16x3 3.3e-5 teacher-forced, 4.2e-4 end to end through
Pipeline.predict; bf16 1.9e-2 (S = 256, every kernel variant within 1.5e-2..1.9e-2).
"""
import numpy as np
import pytest
import torch

import fpnmt_oracle as O

pytestmark = pytest.mark.gpu

BB, L, V, T, B = "mobilenet224_1.0", 2, 512, 12, 3
TOL = {"bf16x3": 2e-3, "bf16": 5e-2}


def _subject_weights():
    w = dict(O.test_weights(BB, vocab=V, layers=L))
    for l in range(L):
        k = "transformer/decoder/dec_layers/%d/mha2/wq/" % l
        w[k + "kernel"] = (w[k + "kernel"] * np.float32(4)).astype(np.float32)
        w[k + "bias"] = (w[k + "bias"] * np.float32(100)).astype(np.float32)
    return w


def _oracle_attention(w, mem, tok):
    with torch.no_grad():
        _, a = O.transformer_logits(mem.double(), tok.long(), O.W(w, torch.float64), O.create_look_ahead_mask(tok.shape[1], torch.float64),
                                    T, num_layers=L)
    return {k: v.cpu() for k, v in a.items()}


_SUBJECTS = {}


def subject(S):
    if S not in _SUBJECTS:
        w = _subject_weights()
        img = O.test_images(B, S, seed=3)
        with torch.no_grad():
            mem = O.encoder(img, O.W(w), BB, num_layers=L, input_vocab_size=(S // 16) ** 2).to(torch.float32)
        tok = torch.randint(4, V, (B, T), generator=torch.Generator().manual_seed(5))
        tok[:, 0] = 2
        ref = _oracle_attention(w, mem, tok)
        wz = dict(w)
        for l in range(L):
            k = "transformer/decoder/dec_layers/%d/mha2/wq/bias" % l
            wz[k] = np.zeros_like(w[k])
        ref_nobias = _oracle_attention(wz, mem, tok)
        nm = (S // 128) ** 2
        for l in range(1, L + 1):                               # the reference is a sharp enough test subject
            c, s = ref["decoder_layer%d_block2" % l], ref["decoder_layer%d_block1" % l]
            assert c.shape[-1] == nm
            assert float(c.amax(-1).mean()) >= 2.0 / nm
            assert float((c - c.roll(1, dims=1)).abs().amax(-1).median()) >= 0.25
            assert float(s.amax(-1).mean()) >= 0.25
            assert float((c - ref_nobias["decoder_layer%d_block2" % l]).abs().max()) >= 0.15
        _SUBJECTS[S] = dict(w=w, mem=mem, tok=tok, ref=ref, nm=nm)
    return _SUBJECTS[S]


def _engine(s, S, beam, prec, opts=(), cache_mode="ancestry", decode_path="chain"):
    from fpnmt.engine import Engine
    return Engine(s["w"], backbone=BB, batch=B, beam=beam, vocab=V, max_len=T, num_layers=L, image_size=S, precision=prec,
                  opts=opts, cache_mode=cache_mode, decode_path=decode_path, use_graphs=False)


def _check_exact_properties(a, nm):
    for k, v in a.items():
        v = v.double()
        assert float((v.sum(-1) - 1).abs().max()) <= 1e-5, k
        if k.endswith("_block1"):
            t = v.shape[-1]
            upper = torch.triu(torch.ones(t, t, dtype=torch.bool), 1)
            assert float(v[..., upper].abs().max()) == 0.0, k        # exact zeros after position t
            assert float(v[:, :, 0, 0].min()) == 1.0, k              # row 0 attends only to <start>
        else:
            assert v.shape[-1] == nm


CASES = [("bf16x3", (), "ancestry"), ("bf16", (), "ancestry"), ("bf16", ("no_xattn",), "ancestry"),
         ("bf16", ("dec_att_simt",), "ancestry"), ("bf16", (), "physical")]
PARAMS = [(prec, opts, cm, S, 4) for prec, opts, cm in CASES for S in (256, 512)] + \
         [(prec, (), "ancestry", S, beam) for prec in ("bf16x3", "bf16") for S in (256, 512) for beam in (1, 16)]


@pytest.mark.parametrize("prec,opts,cache_mode,S,beam", PARAMS)
def test_teacher_forced_attention_matches_oracle(prec, opts, cache_mode, S, beam):
    s = subject(S)
    eng = _engine(s, S, beam, prec, opts, cache_mode)
    a = {k: v.cpu() for k, v in eng.decode_attention(s["mem"].cuda(), s["tok"].int().cuda()).items()}
    eng.close()
    assert sorted(a) == sorted(s["ref"])
    _check_exact_properties(a, s["nm"])
    err = max(float((a[k].double() - s["ref"][k]).abs().max()) for k in a)
    print("%s %s %s S=%d beam=%d: max-abs %.2e" % (prec, opts, cache_mode, S, beam, err))
    assert err <= TOL[prec], err


def test_outputs_are_written_exactly_and_one_may_be_null():
    """Through the raw C ABI: every element of both outputs is written (NaN-filled buffers come back finite), nothing
    after the last memory token of cross_out, and with one output NULL the other is unchanged."""
    S = 256
    s = subject(S)
    eng = _engine(s, S, 4, "bf16")
    tok = s["tok"].int().cuda()
    nm = s["nm"]
    so = torch.full((L, B, 8, T, T), float("nan"), device="cuda")
    co = torch.full((L * B * 8 * T * nm + 64,), float("nan"), device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    from fpnmt import _lib
    _lib.check(eng.lib.fpnmt_decode_attention(eng._h, s["mem"].cuda().data_ptr(), tok.data_ptr(), T, so.data_ptr(), co.data_ptr(), stream))
    torch.cuda.synchronize()
    assert torch.isfinite(so).all() and torch.isfinite(co[:-64]).all() and torch.isnan(co[-64:]).all()
    co2 = torch.full((L, B, 8, T, nm), float("nan"), device="cuda")
    _lib.check(eng.lib.fpnmt_decode_attention(eng._h, None, tok.data_ptr(), T, None, co2.data_ptr(), stream))
    so2 = torch.full((L, B, 8, T, T), float("nan"), device="cuda")
    _lib.check(eng.lib.fpnmt_decode_attention(eng._h, None, tok.data_ptr(), T, so2.data_ptr(), None, stream))
    torch.cuda.synchronize()
    assert float((co2.reshape(-1) - co[:-64]).abs().max()) <= 1e-6 and float((so2 - so).abs().max()) <= 1e-6
    eng.close()


def test_error_paths():
    from fpnmt import _lib
    from fpnmt._lib import FpnmtError
    S = 256
    s = subject(S)
    fused = _engine(s, S, 4, "bf16", decode_path="fused")
    with pytest.raises(FpnmtError) as ei:
        fused.decode_attention(s["mem"].cuda(), s["tok"].int().cuda())
    assert ei.value.code == _lib.ERR_STATE
    fused.close()
    eng = _engine(s, S, 4, "bf16")
    with pytest.raises(FpnmtError) as ei:
        eng.decode_attention(None, torch.zeros(B, T + 1, dtype=torch.int32).cuda())       # t > max_len
    assert ei.value.code == _lib.ERR_INVALID
    tok = s["tok"].int().cuda()
    stream = torch.cuda.current_stream().cuda_stream
    assert eng.lib.fpnmt_decode_attention(eng._h, None, tok.data_ptr(), T, None, None, stream) == _lib.ERR_INVALID
    # DLPack twin: the right shapes work and agree with the raw-pointer entry point; wrong shape / dtype are rejected
    nm = s["nm"]
    mem = s["mem"].cuda()
    ref = eng.decode_attention(mem, tok)
    so, co = torch.zeros(L, B, 8, T, T, device="cuda"), torch.zeros(L, B, 8, T, nm, device="cuda")
    keep = []

    def dl(x):                          # the capsule must outlive the call
        p, k = _lib.dl_tensor(x)
        keep.append(k)
        return p
    assert eng.lib.fpnmt_decode_attention_dl(eng._h, dl(mem), dl(tok), dl(so), dl(co), stream) == 0
    torch.cuda.synchronize()
    assert float((so[1] - ref["decoder_layer2_block1"]).abs().max()) <= 1e-6
    assert float((co[0] - ref["decoder_layer1_block2"]).abs().max()) <= 1e-6
    bad = [(torch.zeros(L, B, 8, T, T + 1, device="cuda"), co), (so, torch.zeros(L, B, 8, T, nm, device="cuda", dtype=torch.float64)),
           (so, torch.zeros(L, B, 8, T, nm + 1, device="cuda")), (torch.zeros(L, B, 8, T, T, device="cuda", dtype=torch.int32), None)]
    for bs, bc in bad:
        assert eng.lib.fpnmt_decode_attention_dl(eng._h, dl(mem), dl(tok), dl(bs), dl(bc) if bc is not None else None, stream) == _lib.ERR_INVALID
    assert eng.lib.fpnmt_decode_attention_dl(eng._h, dl(mem), dl(tok), None, None, stream) == _lib.ERR_INVALID
    eng.close()


def test_launch_accounting():
    """decode_attention adds exactly one probability launch per decoder layer and step to what decode_logits launches."""
    S = 256
    s = subject(S)
    eng = _engine(s, S, 4, "bf16")
    tok = s["tok"][:, :7].int().cuda()
    mem = s["mem"].cuda()
    c0 = eng.launch_count
    eng.decode_logits(mem, tok)
    c1 = eng.launch_count
    eng.decode_attention(mem, tok)
    c2 = eng.launch_count
    eng.close()
    assert (c2 - c1) - (c1 - c0) == L * 7


# ---- captions --------------------------------------------------------------------------------------------------------------
# Pipeline defaults: 512x512 images, 6 layers, beam 4.  With end_bias 56 image 4 of the set ends with <end> after 5 tokens
# and image 0 runs to max_len (checked on the oracle below).
PL, PT, PEND = 6, 12, 56.0


@pytest.fixture(scope="module")
def pipe_subject(tmp_path_factory):
    from fpnmt.dataset import Tokenizer
    from fpnmt.pipeline import Pipeline
    w = O.caption_weights(BB, vocab=V, layers=PL, seed=0, end_bias=PEND)
    img = O.test_images(6, 512, seed=41)[[4, 0]]
    refs = []
    with torch.no_grad():
        mem = O.encoder(img, O.W(w), BB, num_layers=PL, input_vocab_size=(512 // 16) ** 2)
        for i in range(2):
            last = {}
            import fpnmt_oracle.decode as OD
            inner = OD.transformer_logits

            def spy(*a, **kw):
                lg, at = inner(*a, **kw)
                last["attn"] = at
                return lg, at
            OD.transformer_logits = spy
            try:
                res = O.predict_reference(img[i], O.W(w), PT, 4, 2, 3, BB, num_layers=PL, mode="prob", enc_output=mem[i:i + 1])
            finally:
                OD.transformer_logits = inner
            refs.append((res, {k: v[:1].double() for k, v in last["attn"].items()}))
    assert len(refs[0][0]) < PT and len(refs[1][0]) == PT              # one caption ends with <end>, one does not
    pipe = Pipeline(None, None, PT, tokenizer=Tokenizer.synthetic(V), weights=w, beam=4, precision="bf16x3", score_mode="prob")
    return dict(pipe=pipe, img=img, refs=refs)


@pytest.mark.parametrize("i", [0, 1])
def test_predict_plot_layer_returns_the_reference_dict(pipe_subject, i):
    p, (res, ref) = pipe_subject["pipe"], pipe_subject["refs"][i]
    ids, attn = p.predict(pipe_subject["img"][i].numpy(), PT, plot_layer="decoder_layer2_block2")
    assert ids.tolist() == res.tolist()
    n = min(len(res) + 1, PT)
    assert sorted(attn) == sorted(ref)
    for k, v in attn.items():
        assert isinstance(v, np.ndarray) and v.dtype == np.float32
        assert v.shape == ((1, 8, n, n) if k.endswith("_block1") else (1, 8, n, 16)), (k, v.shape)
        err = float(np.abs(v - ref[k].numpy()).max())
        print("predict image %d %s: max-abs %.2e" % (i, k, err))
        assert err <= TOL["bf16x3"], (k, err)
    ids0, none = p.predict(pipe_subject["img"][i].numpy(), PT)
    assert none is None and ids0.tolist() == ids.tolist()


def test_predict_batch_attention_pads_and_matches_single_images(pipe_subject):
    p = pipe_subject["pipe"]
    ids, lens, attn = p.predict_batch(pipe_subject["img"], PT, return_attention=True)
    assert lens[0] != lens[1]
    for i in range(2):
        n = min(int(lens[i]) + 1, PT)
        _, single = p.predict(pipe_subject["img"][i].numpy(), PT, plot_layer=True)
        for k, v in attn.items():
            assert v.shape[:3] == (2, 8, PT)
            assert float(np.abs(v[i, :, n:]).max(initial=0.0)) == 0.0
            if k.endswith("_block1"):
                assert float(np.abs(v[i, :, :, n:]).max(initial=0.0)) == 0.0
                got = v[i:i + 1, :, :n, :n]
            else:
                got = v[i:i + 1, :, :n]
            assert float(np.abs(got - single[k]).max()) <= TOL["bf16x3"], k
