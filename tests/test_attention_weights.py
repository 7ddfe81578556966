"""What the attention weights of a generated caption are, and the host-side construction of the pass that computes them.

The reference's `Pipeline.predict` returns the attention dict of its LAST forward pass (utils/pipeline.py:109-112): the N
beam rows of the prefix before the final top-k.  Under the reference's beam initialisation (all N beams start identical,
pipeline.py:101-102) those rows are one and the same, and they equal the teacher-forced attention of [<start>] + result over
n = len(result) + 1 positions when <end> fired (n = max_seq_len when it did not).  So `Engine.caption_attention` defines a
caption's weights as one teacher-forced pass over its own prefix.  These tests pin that definition on the CPU oracle; the
oracle's `predict_reference` is observed through its `transformer_logits` calls, which return the dict.
"""
import numpy as np
import pytest
import torch

import fpnmt_oracle as O
import fpnmt_oracle.decode as OD
from fpnmt.engine import caption_prefix, mask_caption_attention

BB, S, L, V, T, N = "mobilenet224_1.0", 256, 2, 512, 16, 4


def predict_with_attention(img, w, mem, monkeypatch):
    """predict_reference (beam N, probability scores) and the attention dict of its last forward pass."""
    last = {}
    inner = OD.transformer_logits

    def spy(*a, **kw):
        logits, attn = inner(*a, **kw)
        last["attn"] = attn
        return logits, attn
    monkeypatch.setattr(OD, "transformer_logits", spy)
    res = O.predict_reference(img, O.W(w), T, N, 2, 3, BB, num_layers=L, mode="prob", enc_output=mem)
    monkeypatch.setattr(OD, "transformer_logits", inner)
    return res, last["attn"]


@pytest.fixture(scope="module")
def subject():
    w = O.caption_weights(BB, vocab=V, layers=L, seed=0, end_bias=12.0)
    img = O.test_images(6, S, seed=41)
    with torch.no_grad():
        mem = O.encoder(img, O.W(w), BB, num_layers=L, input_vocab_size=(S // 16) ** 2)
    return w, img, mem


def test_caption_weights_are_one_teacher_forced_pass_over_the_prefix(subject, monkeypatch):
    w, img, mem = subject
    ended = stopped = 0
    with torch.no_grad():
        for i in range(img.shape[0]):
            res, attn = predict_with_attention(img[i], w, mem[i:i + 1], monkeypatch)
            n = min(len(res) + 1, T)                      # <end> fired: len + 1 positions, else all T
            ended += len(res) < T
            stopped += len(res) == T
            tok = torch.tensor([[2] + res.tolist()])[:, :n]
            _, ref = O.transformer_logits(mem[i:i + 1], tok, O.W(w), O.create_look_ahead_mask(n), T, num_layers=L)
            assert sorted(attn) == sorted(ref) == sorted(["decoder_layer%d_block%d" % (l + 1, k) for l in range(L) for k in (1, 2)])
            for k, a in attn.items():
                a = a.to(torch.float64)
                assert a.shape[0] == N and a.shape[2] == n
                assert float((a - a[:1]).abs().max()) == 0.0, k          # the N beam rows are identical
                assert float((a[:1] - ref[k].to(torch.float64)).abs().max()) <= 2e-6, k
    assert ended >= 1 and stopped >= 1, (ended, stopped)               # both kinds of caption are covered


def test_caption_prefix_and_valid_positions():
    ids = torch.tensor([[7, 8, 9, 0, 0], [4, 5, 6, 7, 8], [0, 0, 0, 0, 0], [9, 9, 9, 9, 0]], dtype=torch.int32)
    lens = torch.tensor([3, 5, 0, 4], dtype=torch.int32)
    tok, n = caption_prefix(ids, lens, start_id=2)
    assert tok.dtype == ids.dtype and tok.tolist() == [[2, 7, 8, 9, 0], [2, 4, 5, 6, 7], [2, 0, 0, 0, 0], [2, 9, 9, 9, 9]]
    assert n.tolist() == [4, 5, 1, 5]                                     # min(len + 1, T)


def test_caption_attention_mask_zeroes_rows_and_self_columns():
    B, H, Tn, M = 3, 2, 5, 4
    n = torch.tensor([2, 5, 1])
    attn = {"decoder_layer1_block1": torch.ones(B, H, Tn, Tn), "decoder_layer1_block2": torch.ones(B, H, Tn, M)}
    out = mask_caption_attention(attn, n)
    assert out is attn
    for b in range(B):
        s, c = out["decoder_layer1_block1"][b], out["decoder_layer1_block2"][b]
        k = int(n[b])
        assert float(s[:, :k, :k].min()) == 1.0 and float(s.sum()) == H * k * k
        assert float(c[:, :k].min()) == 1.0 and float(c.sum()) == H * k * M
