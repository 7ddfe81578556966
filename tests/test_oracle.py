"""CPU tests of the oracle itself: TF/Keras op semantics, internal cross-checks (fp32 vs fp64, cached vs uncached
decode, conv vs im2col), and the reference's few numeric anchors (coattention demo inputs, positional encoding)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import fpnmt_oracle as O
from conftest import small_weights


def test_positional_encoding_formula():
    pe = O.raw_positional_encoding(50, 512).numpy()
    pos = np.arange(50)[:, None].astype(np.float64)
    i = np.arange(512)[None, :]
    ang = pos / np.power(10000.0, (2 * (i // 2)) / 512.0)
    ref = np.where(i % 2 == 0, np.sin(ang), np.cos(ang))
    assert np.abs(pe - ref).max() < 1e-6
    assert pe[0, 0] == 0.0 and pe[0, 1] == 1.0                # sin(0), cos(0): interleaved, not concatenated
    assert O.positional_encoding(7, 512).shape == (1, 7, 512)


def test_look_ahead_mask():
    m = O.create_look_ahead_mask(4).numpy()
    assert (m == np.triu(np.ones((4, 4)), 1)).all()


def test_coattention_reference_demo_anchor():
    # models/coattention.py:44-45: all-ones score -> uniform weights 1/49 -> out = hs / 49
    score = torch.ones(1, 1, 7, 7)
    hs = torch.arange(1 * 7 * 7 * 3, dtype=torch.float32).reshape(1, 7, 7, 3).permute(0, 3, 1, 2)
    out = O.coattention_cnn(score, hs)
    assert torch.allclose(out, hs / 49.0, rtol=1e-6)
    # softmax is over ALL positions of an image, independently per image
    s = torch.randn(2, 1, 5, 3)
    w = torch.softmax(s.reshape(2, -1), 1)
    assert torch.allclose(w.sum(1), torch.ones(2), atol=1e-6)


@pytest.mark.parametrize("size,k,stride,expect", [(512, 3, 2, (0, 1)), (256, 3, 2, (0, 1)), (64, 3, 1, (1, 1)),
                                                  (7, 3, 2, (1, 1)), (512, 7, 2, (2, 3)), (8, 2, 2, (0, 0))])
def test_tf_same_padding(size, k, stride, expect):
    assert O.tf_same_pad(size, k, stride) == expect


def test_conv_matches_im2col_with_asymmetric_padding():
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 5, 10, 10, generator=g, dtype=torch.float64)
    k = torch.randn(3, 3, 5, 4, generator=g, dtype=torch.float64)
    y = O.conv2d(x, k, None, 2, ((0, 1), (0, 1)))             # Keras ZeroPadding2D(((0,1),(0,1))) + valid, stride 2
    xp = F.pad(x, (0, 1, 0, 1))
    ref = torch.zeros(2, 4, 5, 5, dtype=torch.float64)
    for oy in range(5):
        for ox in range(5):
            patch = xp[:, :, 2 * oy:2 * oy + 3, 2 * ox:2 * ox + 3]            # (n, c, kh, kw)
            ref[:, :, oy, ox] = torch.einsum("nchw,hwco->no", patch, k)
    assert torch.allclose(y, ref, atol=1e-10)
    assert torch.allclose(O.conv2d(x, k, None, 2, "same"), y)                    # == TF SAME for even sizes


def test_maxpool_same_pads_bottom_right_with_neg_inf():
    x = -torch.ones(1, 1, 4, 4)
    y = O.max_pool(x, 3, 2, "same")
    assert y.shape == (1, 1, 2, 2) and (y == -1).all()        # zero padding would have produced 0


def test_upsample_like_nearest_2x():
    src = torch.arange(6, dtype=torch.float32).reshape(1, 1, 2, 3)
    tgt = torch.zeros(1, 1, 4, 6)
    up = O.upsample_like(src, tgt)
    for y in range(4):
        for x in range(6):
            assert up[0, 0, y, x] == src[0, 0, y // 2, x // 2]


def test_layer_norm_matches_keras_definition():
    x = torch.randn(3, 7, 512)
    g, b = torch.rand(512) + 0.5, torch.randn(512)
    ref = F.layer_norm(x, (512,), g, b, eps=1e-6)
    assert torch.allclose(O.layer_norm(x, g, b, 1e-6), ref, atol=1e-5)


def test_beam_step_ties_lower_flat_index_first():
    # identical rows (the reference's start state): top-N is the arg-max token N times, parents 0..N-1
    n, v = 4, 50
    row = np.random.default_rng(0).normal(size=v).astype(np.float32)
    logits = np.tile(row, (n, 1))
    for mode, s0 in (("prob", np.ones(n, np.float32)), ("log", np.zeros(n, np.float32))):
        parent, token, score = O.beam_step(logits, s0, mode)
        assert parent.tolist() == [0, 1, 2, 3]
        assert (token == row.argmax()).all()
        assert np.allclose(score, score[0])


def test_beam_step_underflow_regime_matches_reference_semantics():
    # once the fp32 probability product is 0 every candidate is 0 and tf.math.top_k returns flat indices 0..N-1
    n, v = 4, 50
    logits = np.random.default_rng(1).normal(size=(n, v)).astype(np.float32)
    parent, token, score = O.beam_step(logits, np.zeros(n, np.float32), "prob")
    assert parent.tolist() == [0, 0, 0, 0] and token.tolist() == [0, 1, 2, 3] and (score == 0).all()


@pytest.mark.parametrize("backbone", ["mobilenet224_1.0", "resnet50", "densenet121"])
def test_backbone_tap_shapes(backbone):
    from fpnmt.weights import BACKBONE_TAPS, init_weights
    w = init_weights(backbone, vocab=64, num_layers=1)
    x = torch.rand(1, 3, 256, 256) * 2 - 1
    c3, c4, c5 = O.backbone_forward(backbone, x, O.W(w))
    ch = BACKBONE_TAPS[backbone]
    assert c3.shape == (1, ch[0], 32, 32) and c4.shape == (1, ch[1], 16, 16) and c5.shape == (1, ch[2], 8, 8)


def test_encoder_shapes_and_view_order():
    w = small_weights("mobilenet224_1.0", 64, 1)
    img = torch.rand(1, 256, 256, 3) * 2 - 1
    taps = {}
    mem = O.encoder(img, O.W(w), num_layers=1, input_vocab_size=256, taps=taps)
    assert [f.shape[1] for f in taps["features"]] == [16, 8, 4, 2, 1]
    assert O.X_ORDER == [0, 1, 2, 4, 3]
    assert [t.shape[1] for t in taps["tokens"]] == [256, 64, 16, 1, 4]          # baseline (P6) last
    assert mem.shape == (1, 4, 512)


def test_fp32_and_fp64_oracles_agree():
    w = small_weights("mobilenet224_1.0", 64, 1)
    img = torch.rand(1, 256, 256, 3, generator=torch.Generator().manual_seed(3)) * 2 - 1
    m32 = O.encoder(img, O.W(w, torch.float32), num_layers=1, input_vocab_size=256)
    m64 = O.encoder(img, O.W(w, torch.float64), num_layers=1, input_vocab_size=256)
    assert (m32.double() - m64).abs().max() < 5e-4


@pytest.mark.parametrize("mode", ["prob", "log"])
def test_cached_batched_decode_equals_faithful_reference_decode(mode):
    """The KV-cached, batched, log-domain decode the engine implements returns exactly what the line-by-line
    restatement of Pipeline.predict returns (no underflow at these lengths)."""
    L, V, T, N = 2, 96, 7, 3
    w = small_weights("mobilenet224_1.0", V, L, seed=5)
    Wv = O.W(w)
    g = torch.Generator().manual_seed(7)
    mem = torch.randn(3, 4, 512, generator=g)
    ids, lens = O.predict_batch_cached(mem, Wv, T, N, 2, 3, num_layers=L)
    for b in range(3):
        ref = O.predict_reference(None, Wv, T, N, 2, 3, num_layers=L, mode=mode, enc_output=mem[b:b + 1])
        assert lens[b] == len(ref)
        assert ids[b, :lens[b]].tolist() == ref.tolist()


def test_end_token_stops_and_is_stripped():
    L, V, T, N = 1, 32, 6, 2
    w = small_weights("mobilenet224_1.0", V, L, seed=9)
    w = dict(w)
    b = w["transformer/final_layer/bias"].copy()
    b[3] = 50.0                                                # <end> always wins
    w["transformer/final_layer/bias"] = b
    mem = torch.randn(2, 4, 512, generator=torch.Generator().manual_seed(1))
    ids, lens = O.predict_batch_cached(mem, O.W(w), T, N, 2, 3, num_layers=L)
    assert lens.tolist() == [0, 0] and (ids == 0).all()        # pipeline.py:147-148 returns beam_result[1:-1] == []
    ref = O.predict_reference(None, O.W(w), T, N, 2, 3, num_layers=L, enc_output=mem[:1])
    assert len(ref) == 0


@pytest.fixture
def at_most_8_threads():
    """With 16 or more threads the CPU GEMM splits the sums of some rows of a 12-row product differently, so rows that are
    equal by construction differ in their last bits; on up to 12 threads they are bit-identical."""
    n = torch.get_num_threads()
    torch.set_num_threads(min(n, 8))
    yield
    torch.set_num_threads(n)


def test_true_beam_extension_explores_and_never_scores_worse_than_greedy(at_most_8_threads):
    """Flagged extension (SURVEY 8f row 4): with only beam 0 alive at t = 0 the first step picks the N best DISTINCT
    tokens of one distribution; on this fixture the returned sequence also scores at least as well as the reference's
    degenerate (N x greedy) search (not a theorem for beam search in general: a fixture property)."""
    L, V, T, N = 2, 96, 6, 4
    w = small_weights("mobilenet224_1.0", V, L, seed=5)
    Wv = O.W(w)
    mem = torch.randn(3, 4, 512, generator=torch.Generator().manual_seed(3))
    tr_true, tr_ref = {}, {}
    ids_t, len_t = O.predict_batch_cached(mem, Wv, T, N, 2, 3, num_layers=L, early_stop=False, trace=tr_true, true_beam=True)
    ids_r, len_r = O.predict_batch_cached(mem, Wv, T, N, 2, 3, num_layers=L, early_stop=False, trace=tr_ref)
    assert ids_t.shape == ids_r.shape and len_t.tolist() == len_r.tolist()
    for b in range(3):
        lg0 = tr_true["logits"][0][b]                          # step-0 logits: all beams fed <start>, rows identical
        assert np.allclose(lg0[0], lg0[1])
        score0 = np.array([0.0] + [-np.inf] * (N - 1), np.float32)
        parent, token, _ = O.beam_step(lg0, score0, "log")
        assert parent.tolist() == [0] * N and len(set(token.tolist())) == N
        assert token.tolist() == np.argsort(-lg0[0], kind="stable")[:N].tolist()

    def seq_logprob(ids_row, b):                               # teacher-forced log-prob of a returned sequence
        toks = torch.tensor([[2] + ids_row.tolist()])
        lp = O.teacher_forced_logprobs(mem[b:b + 1], toks[:, :-1], Wv, T, L)[0]
        return float(sum(lp[i, t] for i, t in enumerate(ids_row.tolist())))
    for b in range(3):
        assert seq_logprob(ids_t[b, :len_t[b]], b) >= seq_logprob(ids_r[b, :len_r[b]], b) - 1e-4
