"""GPU parity of the whole hot path through the C ABI against the CPU oracle.

Per-stage relative L2 error (C3..C5, P3..P7, head outputs, tokens, encoder layers, memory), teacher-forced
log-probs, generated token ids, and size-independent properties at larger sizes.

Tolerances (stated here, checked below):
  BF16X3 parity mode : stage rel-L2 <= 3e-3 ; per-step log-probs within 2e-3 absolute (north-star bound) ;
                       generated token sequences identical to the oracle.
  BF16 fast mode     : a random-init BatchNorm network amplifies perturbations by ~1.2x per layer (rounding every conv
                       operand/output to bf16 in the ORACLE already moves C5 by 40-50 % on these weights), so a fixed
                       stage bound would be meaningless.  The stated bound is relative to that emulation: per stage,
                       rel-L2(engine, oracle) <= max(5e-2 [head outputs: 9e-2], 1.2 x rel-L2(oracle with bf16-rounded
                       convolutions, oracle)).  Measured (profiles/r02_a_parity_stage_errors.json): the engine's error is
                       0.85-1.09 x the emulation's at every tap of the three backbones - it IS the bf16 rounding of this
                       random BatchNorm network, nothing else - and 2-8 % where the network does not amplify (DenseNet).
                       Such a bound cannot see a kernel that is wrong by tens of percent at a few pixels, heads or images:
                       the kernels that run only in this mode (score convolution, stride-1 depthwise, tensor-core encoder
                       attention) and the other encoder bandwidth kernels are held to their own tight bounds, one at a time
                       against fp64 references, in tests/test_gpu_encoder_kernels.py.
                       Decoder (fed with the oracle's memory): log-probs within 0.25 absolute at logit std ~6,
                       per-step arg-max agreement >= 85 %.  Sequence identity is NOT required.
"""
import os

import numpy as np
import pytest
import torch

import fpnmt_oracle as O
from conftest import small_weights

pytestmark = pytest.mark.gpu

B, S, L, V, T, N = 2, 256, 2, 512, 8, 4
BACKBONES = ["resnet50", "mobilenet224_1.0", "densenet121"]


def rel(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _record_stages(bb, prec, table):
    """Measured per-stage errors next to their bounds -> gpurun_out/parity_stages.json (summarised under profiles/)."""
    import json
    d = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    if not os.path.isdir(d):
        return
    p = os.path.join(d, "parity_stages.json")
    data = json.load(open(p)) if os.path.exists(p) else {}
    data["%s/%s" % (bb, prec)] = table
    json.dump(data, open(p, "w"), indent=1, sort_keys=True)


@pytest.fixture(scope="module", params=BACKBONES)
def setup(request):
    bb = request.param
    w = small_weights(bb, V, L)
    Wv = O.W(w)
    img = O.test_images(B, S, seed=1)
    taps = {}
    mem_ref = O.encoder(img, Wv, bb, num_layers=L, input_vocab_size=(S // 16) ** 2, taps=taps)
    taps_emu = {}
    with O.bf16_conv_emulation():
        mem_emu = O.encoder(img, Wv, bb, num_layers=L, input_vocab_size=(S // 16) ** 2, taps=taps_emu)
    return dict(bb=bb, w=w, Wv=Wv, img=img, taps=taps, mem_ref=mem_ref, taps_emu=taps_emu, mem_emu=mem_emu)


@pytest.mark.parametrize("prec,tol", [("bf16x3", 3e-3), ("bf16", 5e-2)])
def test_encoder_stages(setup, prec, tol):
    from fpnmt.engine import Engine
    s = setup
    eng = Engine(s["w"], backbone=s["bb"], batch=B, beam=N, vocab=V, max_len=T, num_layers=L, image_size=S,
                 precision=prec, use_graphs=False)
    mem = eng.encode(s["img"].cuda())
    taps, emu = s["taps"], s["taps_emu"]
    errs, bound = {}, {}

    def check(key, got, ref, ref_emu):
        errs[key] = rel(got.cpu().reshape(ref.shape), ref)
        base = tol * (1.5 if prec == "bf16x3" else 1.8) if key.startswith("feat") else tol
        bound[key] = base if prec == "bf16x3" else max(base, 1.2 * rel(ref_emu, ref))

    for nm in ("C3", "C4", "C5", "P3", "P4", "P5", "P6", "P7"):
        check(nm, eng.tap(nm), taps[nm], emu[nm])
    for i in range(5):
        check("feat%d" % i, eng.tap("feat%d" % i), taps["features"][i], emu["features"][i])
        check("tokens%d" % i, eng.tap("tokens%d" % i), taps["tokens"][i], emu["tokens"][i])
    for l in range(L):
        check("enc_layer%d" % l, eng.tap("enc_layer%d" % l), taps["enc_layer%d" % l], emu["enc_layer%d" % l])
    check("memory", mem, s["mem_ref"], s["mem_emu"])
    feats = eng.features(s["img"].cuda())
    for i in range(5):
        assert tuple(feats[i].shape) == tuple(taps["features"][i].shape)
        check("features_api%d" % i, feats[i], taps["features"][i], emu["features"][i])
    eng.close()
    print("%s %s stage rel-L2 (bound): " % (s["bb"], prec) + "  ".join("%s %.2e (%.2e)" % (k, errs[k], bound[k]) for k in errs))
    _record_stages(s["bb"], prec, {k: {"err": errs[k], "bound": bound[k]} for k in errs})
    bad = {k: (v, bound[k]) for k, v in errs.items() if not v < bound[k]}
    assert not bad, (s["bb"], prec, bad)


@pytest.mark.parametrize("prec", ["bf16x3", "bf16"])
def test_teacher_forced_logprobs_and_generate(setup, prec):
    from fpnmt.engine import Engine
    s = setup
    eng = Engine(s["w"], backbone=s["bb"], batch=B, beam=N, vocab=V, max_len=T, num_layers=L, image_size=S,
                 precision=prec, use_graphs=True)
    gtok = torch.randint(4, V, (B, T), generator=torch.Generator().manual_seed(2))
    gtok[:, 0] = 2
    lg = eng.decode_logits(s["mem_ref"].cuda(), gtok.int().cuda()).cpu()
    ref_lg, _ = O.transformer_logits(s["mem_ref"], gtok, s["Wv"], O.create_look_ahead_mask(T), T, num_layers=L)
    lp, lpr = torch.log_softmax(lg, -1), torch.log_softmax(ref_lg, -1)
    err = float((lp - lpr).abs().max())
    agree = float((lp.argmax(-1) == lpr.argmax(-1)).float().mean())
    ids, lens = eng.generate(s["img"].cuda(), early_stop=True)
    ref_ids, ref_len = O.predict_batch_cached(s["mem_ref"], s["Wv"], T, N, 2, 3, num_layers=L)
    eng.close()
    if prec == "bf16x3":
        assert err < 2e-3, err                                   # north-star: per-step log-probs within 2e-3 absolute
        assert agree == 1.0
        assert (ids.numpy() == ref_ids).all() and (lens.numpy() == ref_len).all()
    else:
        assert err < 0.25 and agree >= 0.85, (err, agree)        # bf16-mode tolerance, stated separately


def test_generate_matches_faithful_reference_loop_prob_scores():
    """Engine in the reference's own score domain (product of probabilities) vs the line-by-line restatement of
    Pipeline.predict (uncached, per image)."""
    from fpnmt.engine import Engine
    bb = "mobilenet224_1.0"
    w = small_weights(bb, V, L, seed=11)
    Wv = O.W(w)
    img = O.test_images(B, S, seed=5)
    eng = Engine(w, backbone=bb, batch=B, beam=N, vocab=V, max_len=T, num_layers=L, image_size=S, precision="bf16x3",
                 score_mode="prob", use_graphs=True)
    ids, lens = eng.generate(img.cuda(), early_stop=True)
    eng.close()
    for b in range(B):
        ref = O.predict_reference(img[b], Wv, T, N, 2, 3, bb, num_layers=L, mode="prob")
        assert lens[b] == len(ref) and ids[b, :lens[b]].tolist() == ref.tolist()


def test_end_token_early_stop_and_strip():
    from fpnmt.engine import Engine
    bb = "mobilenet224_1.0"
    w = dict(small_weights(bb, V, L, seed=3))
    b = w["transformer/final_layer/bias"].copy()
    b[3] = 60.0
    w["transformer/final_layer/bias"] = b
    img = O.test_images(B, S, seed=6)
    eng = Engine(w, backbone=bb, batch=B, beam=N, vocab=V, max_len=T, num_layers=L, image_size=S, precision="bf16x3")
    ids, lens = eng.generate(img.cuda(), early_stop=True)
    ids2, lens2 = eng.generate(img.cuda(), early_stop=False)       # fixed-length run freezes finished images
    eng.close()
    assert lens.tolist() == [0, 0] and (ids == 0).all()
    assert lens2.tolist() == [0, 0] and (ids2 == 0).all()


def test_batch_invariance_and_determinism_512():
    """Size-independent properties at the full 512x512 resolution: captions and memory do not depend on the batch
    position or on the other images of the batch; repeated runs are bit-identical; graphs == eager."""
    from fpnmt.engine import Engine
    from fpnmt.weights import init_weights
    bb, Bf, Nf, Vf, Tf = "mobilenet224_1.0", 4, 8, 1000, 12
    w = small_weights(bb, Vf, 2, seed=2)
    imgs = O.test_images(Bf, 512, seed=9)
    eng = Engine(w, backbone=bb, batch=Bf, beam=Nf, vocab=Vf, max_len=Tf, num_layers=2, image_size=512, use_graphs=True)
    eng2 = Engine(w, backbone=bb, batch=Bf, beam=Nf, vocab=Vf, max_len=Tf, num_layers=2, image_size=512, use_graphs=False)
    m1 = eng.encode(imgs.cuda()).cpu()
    ids1, len1 = eng.generate(imgs.cuda(), early_stop=False)
    ids1b, len1b = eng.generate(imgs.cuda(), early_stop=False)
    perm = torch.tensor([2, 0, 3, 1])
    m2 = eng.encode(imgs[perm].cuda()).cpu()
    ids2, len2 = eng.generate(imgs[perm].cuda(), early_stop=False)
    ids3, len3 = eng2.generate(imgs.cuda(), early_stop=False)
    assert m1.shape == (Bf, 16, 512)
    assert torch.equal(ids1, ids1b) and torch.equal(len1, len1b)
    assert torch.equal(m1[perm], m2)
    assert torch.equal(ids1[perm], ids2) and torch.equal(len1[perm], len2)
    assert torch.equal(ids1, ids3) and torch.equal(len1, len3)
    assert int(len1.min()) >= 1 and int(ids1.max()) < Vf
    eng.close(); eng2.close()


def test_pipeline_mirror_end_to_end(tmp_path):
    """Reference-facing API: Pipeline(tokenizer_filename, checkpoint_path, max_seq_len).evaluate_img / evaluate."""
    from fpnmt.dataset import Tokenizer, store_tokenizer_to_path
    from fpnmt.pipeline import Pipeline
    from fpnmt.weights import save_weights
    vocab = 300
    tok_path = str(tmp_path / "_tokenizer.json")
    store_tokenizer_to_path(Tokenizer.synthetic(vocab), tok_path)
    w = small_weights("mobilenet224_1.0", vocab, 6, seed=4)
    save_weights(str(tmp_path / "weights.npz"), w)
    pipe = Pipeline(tok_path, str(tmp_path), 10, beam=4)
    assert pipe.target_vocab_size == vocab and pipe.max_seq_len == 10
    img = O.test_images(1, 512, seed=8)[0].numpy()
    ids, attn = pipe.predict(img, 10)
    assert attn is None and ids.ndim == 1 and len(ids) <= 10
    res = pipe.evaluate_img(img, 10)
    assert res[0]["image_id"] == 0 and isinstance(res[0]["caption"], str)
    assert res[0]["caption"] == pipe.tokenizer.sequences_to_texts([ids])[0]
    res2 = pipe.evaluate([(img, 17), (img, 18), (img, 19)], 10, batch_size=2)
    assert [r["image_id"] for r in res2] == [17, 18, 19] and all(r["caption"] == res[0]["caption"] for r in res2)
    # the same through three lanes (batches in flight on the GPU): same rows, same order
    imgs7 = [(O.test_images(1, 512, seed=20 + i)[0].numpy(), 100 + i) for i in range(7)]
    rows3 = pipe.evaluate(imgs7, 10, batch_size=2, lanes=3)
    assert [r["image_id"] for r in rows3] == [100 + i for i in range(7)]
    assert rows3 == pipe.evaluate(imgs7, 10, batch_size=2, lanes=2)        # (lanes >= 2 share one kernel set)
    # Transformer.call parity surface: logits for a teacher-forced prefix
    mem = pipe.transformer.encoder(torch.from_numpy(img)[None], False, None)
    logits, _ = pipe.transformer(mem, torch.tensor([[2, 5, 9]]), False, None)
    assert tuple(logits.shape) == (1, 3, vocab + (-vocab) % 8)


def test_engine_matches_reference_goldens():
    """CUDA engine vs the golden vectors recorded from the reference's OWN modules (tests/golden/make_golden.py):
    FeatureExtractor.call outputs, Encoder.call memory and Pipeline.predict token ids (beam 4 and 8)."""
    import os
    from fpnmt.engine import Engine
    with np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_model.npz")) as z:
        gold = {k: z[k] for k in z.files}
    Lg, Vg, Tg, Sg = (int(v) for v in gold["fe_cfg"])
    w = O.test_weights("mobilenet224_1.0", vocab=Vg, layers=Lg, seed=0)
    img = O.test_images(2, Sg, seed=int(gold["fe_image_seed"][0]))
    for beam in (4, 8):
        eng = Engine(w, backbone="mobilenet224_1.0", batch=2, beam=beam, vocab=Vg, max_len=Tg, num_layers=Lg, image_size=Sg,
                     precision="bf16x3", score_mode="prob", use_graphs=True)
        if beam == 4:
            feats = eng.features(img.cuda())
            for i in range(5):
                assert rel(feats[i][:1].cpu(), torch.from_numpy(gold["fe_feat%d" % i])) < 3e-3, i
            mem = eng.encode(img.cuda()).cpu()
            assert rel(mem, torch.from_numpy(gold["fe_memory"])) < 3e-3
            assert float((mem - torch.from_numpy(gold["fe_memory"])).abs().max()) < 2e-2
        ids, lens = eng.generate(img.cuda(), early_stop=True)
        for i in range(2):
            assert ids[i, :lens[i]].tolist() == gold["predict_beam%d_img%d" % (beam, i)].tolist(), (beam, i)
        eng.close()


def test_encoder_attention_mma_matches_simt_path():
    """bf16 mode: the mma.sync flash kernel of the encoder's cross-level attention vs the fp32 CUDA-core kernel on the
    same bf16 K/V/Q (the only differences are P rounded to bf16 and the summation order): encoder layers within 2e-2."""
    import os
    from fpnmt.engine import Engine
    bb = "mobilenet224_1.0"
    w = small_weights(bb, V, L, seed=7)
    img = O.test_images(B, 512, seed=4)           # 512x512: the P3 view has 1024 keys (16 tiles of 64)
    outs = {}
    for mode in ("0", "1"):
        eng = Engine(w, backbone=bb, batch=B, beam=N, vocab=V, max_len=T, num_layers=L, image_size=512, precision="bf16",
                     use_graphs=False, opts=("enc_att_simt",) if mode == "1" else ())
        eng.encode(img.cuda())
        outs[mode] = [eng.tap("enc_layer%d" % l).cpu() for l in range(L)]
        eng.close()
    for l in range(L):
        assert rel(outs["0"][l], outs["1"][l]) < 2e-2, (l, rel(outs["0"][l], outs["1"][l]))


@pytest.mark.parametrize("size", [512, 256])
def test_fused_cross_attention_block_matches_unfused_path(size):
    """bf16 mode: xattn_kernel (folded Q/O projections + softmax over the memory tokens + residual + LayerNorm in one
    tcgen05 kernel) vs the three separate kernels on the same weights / memory / tokens.  512x512 has 16 memory tokens,
    256x256 has 4 (exercises the padded-token mask).  Differences: the folded operands are rounded to bf16 once more and
    P is bf16 -> teacher-forced logits within 5e-2 relative L2, arg-max agreement >= 90 %."""
    import os
    from fpnmt.engine import Engine
    bb = "mobilenet224_1.0"
    w = small_weights(bb, V, L, seed=12)
    img = O.test_images(B, size, seed=3)
    gtok = torch.randint(4, V, (B, T), generator=torch.Generator().manual_seed(5))
    gtok[:, 0] = 2
    outs = {}
    for mode in ("1", "0"):
        eng = Engine(w, backbone=bb, batch=B, beam=N, vocab=V, max_len=T, num_layers=L, image_size=size, precision="bf16",
                     use_graphs=False, decode_path="chain", opts=() if mode == "1" else ("no_xattn",))
        eng.encode(img.cuda())
        outs[mode] = eng.decode_logits(None, gtok.int().cuda()).cpu()
        ids, lens = eng.generate(img.cuda(), early_stop=False)
        outs["ids" + mode] = ids.clone()
        eng.close()
    err = rel(outs["1"], outs["0"])
    agree = float((outs["1"].argmax(-1) == outs["0"].argmax(-1)).float().mean())
    assert err < 5e-2 and agree >= 0.9, (size, err, agree)
    assert torch.isfinite(outs["1"]).all()


def test_c1_greedy_single_image_resnet50_matches_faithful_reference_loop():
    """BASELINE config C1 shape: ResNet-50-FPN, greedy (beam 1), batch 1, 512x512 — token ids identical to the
    line-by-line restatement of Pipeline.predict (uncached, probability-product scores)."""
    from fpnmt.engine import Engine
    bb = "resnet50"
    w = small_weights(bb, V, L, seed=21)
    img = O.test_images(1, 512, seed=13)
    eng = Engine(w, backbone=bb, batch=1, beam=1, vocab=V, max_len=T, num_layers=L, image_size=512, precision="bf16x3",
                 score_mode="prob", use_graphs=True)
    ids, lens = eng.generate(img.cuda(), early_stop=True)
    eng.close()
    ref = O.predict_reference(img[0], O.W(w), T, 1, 2, 3, bb, num_layers=L, mode="prob")
    assert lens[0] == len(ref) and ids[0, :lens[0]].tolist() == ref.tolist()


@pytest.mark.parametrize("beam", [3, 16])
def test_fused_cross_attention_other_beam_widths(beam):
    """xattn_kernel pads the beam rows of an image to 16 MMA columns: odd and maximal widths vs the unfused path."""
    from fpnmt.engine import Engine
    bb = "mobilenet224_1.0"
    w = small_weights(bb, V, L, seed=14)
    img = O.test_images(3, 256, seed=2)
    gtok = torch.randint(4, V, (3, T), generator=torch.Generator().manual_seed(6))
    gtok[:, 0] = 2
    outs = {}
    for mode in ("1", "0"):
        eng = Engine(w, backbone=bb, batch=3, beam=beam, vocab=V, max_len=T, num_layers=L, image_size=256,
                     precision="bf16", use_graphs=False, decode_path="chain", opts=() if mode == "1" else ("no_xattn",))
        eng.encode(img.cuda())
        outs[mode] = eng.decode_logits(None, gtok.int().cuda()).cpu()
        ids, lens = eng.generate(img.cuda(), early_stop=False)
        outs["ids" + mode] = ids
        eng.close()
    assert rel(outs["1"], outs["0"]) < 5e-2
    assert (outs["ids1"] == outs["ids0"]).float().mean() >= 0.7


def test_engine_error_paths():
    """The C ABI reports misuse through error codes / FpnmtError; nothing falls back silently."""
    from fpnmt._lib import FpnmtError
    from fpnmt.engine import Engine
    bb = "mobilenet224_1.0"
    w = dict(small_weights(bb, V, L, seed=1))
    eng = Engine(w, backbone=bb, batch=B, beam=N, vocab=V, max_len=T, num_layers=L, image_size=256)
    with pytest.raises(ValueError):
        eng.encode(torch.zeros(B, 128, 128, 3).cuda())                     # wrong spatial size
    with pytest.raises(FpnmtError):
        eng.decode_logits(None, torch.zeros(B, T + 5, dtype=torch.int32).cuda())   # t > max_len
    with pytest.raises(FpnmtError):
        eng.tap("no_such_layer")
    eng.close()
    w.pop("transformer/final_layer/kernel")
    with pytest.raises(FpnmtError) as ei:
        Engine(w, backbone=bb, batch=B, beam=N, vocab=V, max_len=T, num_layers=L, image_size=256)
    assert "final_layer" in str(ei.value)
    with pytest.raises(FpnmtError):
        Engine(small_weights(bb, V, L, seed=1), backbone=bb, batch=B, beam=64, vocab=V, max_len=T, num_layers=L, image_size=256)
    # malformed weights are rejected by name instead of being read or written out of bounds (ADVICE r01)
    FE = "transformer/encoder/feature_extractor/retinanet_model"
    for key, bad, needle in (
            (FE + "/P4/bias", np.zeros(255, np.float32), "P4/bias"),                                   # short bias vector
            (FE + "/P4/kernel", np.zeros((3, 3, 256, 264), np.float32), "P4"),                         # more filters than the layer
            (FE + "/bn_Conv1/gamma", np.zeros(16, np.float32), "bn_Conv1"),                            # BatchNorm vector too short
            ("transformer/decoder/dec_layers/0/ffn1/bias", np.zeros(100, np.float32), "ffn1/bias"),
            ("transformer/decoder/dec_layers/0/mha1/wq/kernel", np.zeros((512, 520), np.float32), "")):  # Dense with extra outputs
        wb = dict(small_weights(bb, V, L, seed=1))
        assert key in wb, key
        wb[key] = bad
        with pytest.raises(FpnmtError) as ei:
            Engine(wb, backbone=bb, batch=B, beam=N, vocab=V, max_len=T, num_layers=L, image_size=256)
        assert needle in str(ei.value), (key, str(ei.value))
    with pytest.raises(FpnmtError):
        Engine(small_weights(bb, V, L, seed=1), backbone=bb, batch=B, beam=N, vocab=V, max_len=T, num_layers=L, image_size=300)


def test_double_buffered_host_input_matches_one_shot_generate():
    """fpnmt_stage_images + fpnmt_generate_staged (Engine.generate_stream): same captions as the one-shot call for
    every batch of a stream, in order, including a stream of one batch; an empty slot is a state error."""
    from fpnmt._lib import FpnmtError
    from fpnmt.engine import Engine
    bb = "mobilenet224_1.0"
    w = small_weights(bb, V, L, seed=4)
    eng = Engine(w, backbone=bb, batch=B, beam=N, vocab=V, max_len=T, num_layers=L, image_size=S, precision="bf16x3")
    batches = [O.test_images(B, S, seed=30 + i).pin_memory() for i in range(5)]
    want = [eng.generate(b, early_stop=False) for b in batches]
    got = list(eng.generate_stream(iter(batches), early_stop=False))
    assert len(got) == 5
    for (i0, l0), (i1, l1) in zip(want, got):
        assert torch.equal(i0, i1) and torch.equal(l0, l1)
    one = list(eng.generate_stream([batches[2].numpy()], early_stop=True))       # pageable numpy input, early stop
    ref_ids, ref_len = eng.generate(batches[2], early_stop=True)
    assert len(one) == 1 and torch.equal(one[0][0], ref_ids) and torch.equal(one[0][1], ref_len)
    assert list(eng.generate_stream([], early_stop=True)) == []
    with pytest.raises(FpnmtError):
        eng.generate_staged(1)
    with pytest.raises(ValueError):
        eng.stage(torch.zeros(B, S, S, 3).cuda(), 0)
    eng.close()


def test_config_words_that_select_nothing_are_refused():
    """fpnmt_create refuses a dec_groups above 1, a kernel_opts bit that no FPNMT_OPT_* defines (16 and 64 included) and a
    non-zero reserved word with FPNMT_ERR_INVALID and a message, instead of silently building the default engine."""
    import ctypes as C
    from fpnmt import _lib
    lib = _lib.load()

    def create(**words):
        c = _lib.FpnmtConfig()
        c.backbone, c.image_size, c.batch, c.beam, c.vocab, c.max_len = 0, S, B, N, V, T
        c.num_layers, c.d_model, c.num_heads, c.dff, c.start_id, c.end_id = L, 512, 8, 2048, 2, 3
        for k, v in words.items():
            if k == "reserved0":
                c.reserved[0] = v
            else:
                setattr(c, k, v)
        h = C.c_void_p()
        rc = lib.fpnmt_create(C.byref(c), 0, C.byref(h))
        msg = lib.fpnmt_last_error().decode()
        if rc == _lib.OK:
            lib.fpnmt_destroy(h)
        return rc, msg

    assert create(dec_groups=1)[0] == _lib.OK
    for words, word in (({"dec_groups": 2}, "dec_groups"), ({"kernel_opts": 16}, "kernel_opts"), ({"kernel_opts": 64}, "kernel_opts"),
                        ({"reserved0": 1}, "reserved")):
        rc, msg = create(**words)
        assert rc == _lib.ERR_INVALID and word in msg, (words, rc, msg)


@pytest.mark.parametrize("bb", BACKBONES)
def test_fused_stem_matches_im2col_path(bb):
    """stem_kernel (image -> im2col tile built in shared memory -> tcgen05) vs the explicit im2col + GEMM stem: same bf16
    operands and fp32 accumulation, only the summation order differs, so the first backbone taps agree to bf16 rounding."""
    from fpnmt.engine import Engine
    w = small_weights(bb, V, L, seed=5)
    img = O.test_images(3, 512, seed=17).cuda()
    taps = {}
    for mode in ("1", "0"):
        eng = Engine(w, backbone=bb, batch=3, beam=N, vocab=V, max_len=T, num_layers=L, image_size=512, precision="bf16",
                     use_graphs=False, opts=() if mode == "1" else ("no_stem",))
        eng.encode(img)
        taps[mode] = {n: eng.tap(n).cpu() for n in ("C3", "C5", "P3")}
        eng.close()
    assert rel(taps["1"]["C3"], taps["0"]["C3"]) < 1e-2
    assert rel(taps["1"]["P3"], taps["0"]["P3"]) < 3e-2
    assert torch.isfinite(taps["1"]["C5"]).all()


def test_true_beam_extension_matches_oracle():
    """true_beam=1 (flagged extension, SURVEY 8f row 4): only beam 0 alive at t = 0, so the beams diverge.  Same ids as
    the oracle's cached decode with the same initial scores (BF16X3 mode, log scores)."""
    from fpnmt.engine import Engine
    bb = "mobilenet224_1.0"
    w = small_weights(bb, V, L, seed=23)
    Wv = O.W(w)
    img = O.test_images(B, S, seed=31)
    mem = O.encoder(img, Wv, bb, num_layers=L, input_vocab_size=(S // 16) ** 2)
    ref_ids, ref_len = O.predict_batch_cached(mem, Wv, T, N, 2, 3, num_layers=L, early_stop=False, true_beam=True)
    greedy_ids, _ = O.predict_batch_cached(mem, Wv, T, N, 2, 3, num_layers=L, early_stop=False)
    eng = Engine(w, backbone=bb, batch=B, beam=N, vocab=V, max_len=T, num_layers=L, image_size=S, precision="bf16x3",
                 true_beam=True)
    ids, lens = eng.generate(img.cuda(), early_stop=False)
    eng.close()
    assert lens.tolist() == ref_len.tolist()
    assert ids.numpy().tolist() == ref_ids.tolist()
    # the extension is not a no-op: a real beam may (and here does, for at least one image or step) leave the greedy path,
    # and its final score is never worse; identical output is also legal, so only the shapes are asserted unconditionally
    assert ids.shape == greedy_ids.shape


def test_c2_full_size_properties():
    """BASELINE config C2 at FULL size (ResNet-50-FPN, batch 64, beam 8, V = 10 000, T = 64, 6 layers, 512x512, the bench's
    weight factory): size-independent properties - repeated runs bit-identical, captions follow their images under a batch
    permutation, the streaming (double-buffered) call equals the one-shot call, and a 4-image engine built from the same
    weights reproduces the first images of the 64-image batch (batch-size invariance of every kernel's tiling)."""
    from fpnmt.engine import Engine
    from fpnmt.weights import init_weights
    bb, Bf, Nf, Vf, Tf = "resnet50", 64, 8, 10000, 64
    w = init_weights(bb, vocab=Vf, seed=0)
    g = torch.Generator().manual_seed(1234)
    imgs = (torch.rand(Bf, 512, 512, 3, generator=g) * 2 - 1)
    eng = Engine(w, backbone=bb, batch=Bf, beam=Nf, vocab=Vf, max_len=Tf, use_graphs=True)
    dev = imgs.cuda()
    ids1, len1 = eng.generate(dev, early_stop=False)
    ids1b, len1b = eng.generate(dev, early_stop=False)
    assert torch.equal(ids1, ids1b) and torch.equal(len1, len1b)
    assert tuple(ids1.shape) == (Bf, Tf) and int(len1.min()) == Tf and int(ids1.max()) < Vf and int(ids1.min()) >= 0
    perm = torch.randperm(Bf, generator=torch.Generator().manual_seed(5))
    ids2, len2 = eng.generate(imgs[perm].cuda(), early_stop=False)
    assert torch.equal(ids1[perm], ids2) and torch.equal(len1[perm], len2)
    pinned = [imgs.pin_memory(), imgs[perm].contiguous().pin_memory()]
    outs = list(eng.generate_stream(iter(pinned), early_stop=False))
    assert torch.equal(outs[0][0], ids1) and torch.equal(outs[1][0], ids2)
    eng.close()
    small = Engine(w, backbone=bb, batch=4, beam=Nf, vocab=Vf, max_len=Tf, use_graphs=True)
    ids4, len4 = small.generate(imgs[:4].cuda(), early_stop=False)
    small.close()
    assert torch.equal(ids4, ids1[:4]) and torch.equal(len4, len1[:4])


def test_full_depth_resnet50_512_parity_bf16x3():
    """The reference's own depth and resolution (ResNet-50-FPN, 512x512, 6 encoder + 6 decoder layers) in the parity
    mode: encoder memory within 3e-3 rel-L2 of the oracle, teacher-forced per-step log-probs within the north-star 2e-3
    absolute, arg-max identical, generated ids identical to the oracle's cached decode."""
    from fpnmt.engine import Engine
    bb, Lf, Vf, Tf, Nf = "resnet50", 6, 1000, 8, 4
    w = small_weights(bb, Vf, Lf, seed=3)
    Wv = O.W(w)
    img = O.test_images(1, 512, seed=21)
    with torch.no_grad():
        mem_ref = O.encoder(img, Wv, bb, num_layers=Lf, input_vocab_size=1024)
    eng = Engine(w, backbone=bb, batch=1, beam=Nf, vocab=Vf, max_len=Tf, num_layers=Lf, image_size=512, precision="bf16x3")
    mem = eng.encode(img.cuda()).cpu()
    assert rel(mem, mem_ref) < 3e-3
    gtok = torch.randint(4, Vf, (1, Tf), generator=torch.Generator().manual_seed(8))
    gtok[:, 0] = 2
    lg = eng.decode_logits(mem_ref.cuda(), gtok.int().cuda()).cpu()
    ref_lg, _ = O.transformer_logits(mem_ref, gtok, Wv, O.create_look_ahead_mask(Tf), Tf, num_layers=Lf)
    lp, lpr = torch.log_softmax(lg, -1), torch.log_softmax(ref_lg, -1)
    assert float((lp - lpr).abs().max()) < 2e-3
    assert bool((lp.argmax(-1) == lpr.argmax(-1)).all())
    ids, lens = eng.generate(img.cuda(), early_stop=True)
    ref_ids, ref_len = O.predict_batch_cached(mem_ref, Wv, Tf, Nf, 2, 3, num_layers=Lf)
    eng.close()
    assert (ids.numpy() == ref_ids).all() and (lens.numpy() == ref_len).all()


def test_two_engines_on_two_devices_in_one_process():
    """Opt-in shared-memory sizes are per-device function attributes (ADVICE r01): a second engine on another GPU of the
    same process must launch every kernel (k_enc_attention_mma 66 KB, k_conv3x3_c1 57 KB, k_beam_step) and agree with
    the first one bit for bit."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from fpnmt.engine import Engine
    bb = "mobilenet224_1.0"
    w = small_weights(bb, V, L, seed=6)
    img = O.test_images(B, S, seed=14)
    outs = []
    for dev in (1, 0):            # device 1 FIRST: a once-per-process guard would have armed device 0 only
        with torch.cuda.device(dev):
            eng = Engine(w, backbone=bb, batch=B, beam=N, vocab=V, max_len=T, num_layers=L, image_size=S, precision="bf16",
                         device=dev)
            ids, lens = eng.generate(img.to("cuda:%d" % dev), early_stop=False)
            torch.cuda.synchronize(dev)
            outs.append((ids.clone(), lens.clone()))
            eng.close()
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
