"""Caption parity on 100 images whose captions are NOT degenerate (VERDICT r01 "next" #1).

`fpnmt_oracle.caption_weights` gives greedy captions with ~12 distinct tokens each, all 100 different, ~10 % of them
ending early with <end>, and a true beam search that leaves the greedy path on ~90 % of the images - so beam reorder,
the ancestry table, mid-sequence <end> and the per-image early stop are all exercised end to end.  Asserted here:

  BF16X3 (fp32-class parity mode)  sequence identity with the oracle on >= 99 % of the images (north-star bound), for the
                                   reference's beam initialisation AND for the true-beam extension; teacher-forced per-step
                                   log-probs within 2e-3 absolute on the oracle's own captions.
  BF16 (the benchmarked mode)      the measured numbers are printed and written to gpurun_out/parity_captions.json:
                                   sequence identity end to end (bf16 CNN + bf16 decoder) and decoder-only (fed with the
                                   oracle's memory), per-step arg-max agreement and log-prob error teacher-forced on the
                                   oracle's captions.  Stated tolerance: per-step agreement >= 95 %, log-probs within 1.0
                                   absolute at logit std 5 (logits up to +-25), decoder-only sequence identity >= 50 % (a
                                   caption is lost at its first flipped step; the median top-1/top-2 margin of these weights
                                   is ~0.5 nat).  End-to-end identity is reported, not asserted: bf16 storage of the CNN
                                   activations moves this random-BatchNorm network's memory by ~20 % (tests/test_gpu_engine.py
                                   holds that to the bf16-rounding emulation of the oracle), which changes most captions.
"""
import json
import os

import numpy as np
import pytest
import torch

import fpnmt_oracle as O

pytestmark = pytest.mark.gpu

BB, S, L, V, T, N = "mobilenet224_1.0", 256, 2, 1000, 16, 8
NIMG, BATCH = 100, 20
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _record(key, value):
    d = os.path.join(ROOT, "gpurun_out")
    if not os.path.isdir(d):
        return
    p = os.path.join(d, "parity_captions.json")
    data = {}
    if os.path.exists(p):
        try:
            data = json.load(open(p))
        except Exception:
            data = {}
    data[key] = value
    json.dump(data, open(p, "w"), indent=1, sort_keys=True)


@pytest.fixture(scope="module")
def subject():
    w = O.caption_weights(BB, vocab=V, layers=L, seed=0, end_bias=6.0)
    Wv = O.W(w)
    img = O.test_images(NIMG, S, seed=41)
    with torch.no_grad():
        mem = O.encoder(img, Wv, BB, num_layers=L, input_vocab_size=(S // 16) ** 2)
    ids, lens = O.predict_batch_cached(mem, Wv, T, N, 2, 3, num_layers=L, early_stop=True)
    ids_tb, lens_tb = O.predict_batch_cached(mem, Wv, T, N, 2, 3, num_layers=L, early_stop=True, true_beam=True)
    return dict(w=w, Wv=Wv, img=img, mem=mem, ids=ids, lens=lens, ids_tb=ids_tb, lens_tb=lens_tb)


def test_oracle_captions_are_not_degenerate(subject):
    s = subject
    distinct = np.array([len(set(r[:n].tolist())) for r, n in zip(s["ids"], s["lens"])])
    assert (distinct >= 5).mean() >= 0.95, distinct
    assert len(set(tuple(r.tolist()) for r in s["ids"])) >= 90                    # captions depend on the image
    assert ((s["lens"] < T).sum() >= 5) and ((s["lens"] == T).sum() >= 50)         # <end> fires mid-sequence on some
    differs = (s["ids"] != s["ids_tb"]).any(axis=1) | (s["lens"] != s["lens_tb"])
    assert differs.mean() >= 0.5                                                  # a true beam leaves the greedy path


def _same(ids, lens, ref_ids, ref_lens):
    return (np.asarray(ids) == ref_ids).all(axis=1) & (np.asarray(lens) == ref_lens)


def _run(s, prec, true_beam=False, opts=()):
    from fpnmt.engine import Engine
    eng = Engine(s["w"], backbone=BB, batch=BATCH, beam=N, vocab=V, max_len=T, num_layers=L, image_size=S, precision=prec,
                 true_beam=true_beam, use_graphs=True, opts=opts)
    e2e_ids, e2e_lens, dec_ids, dec_lens, lp_err, agree, steps = [], [], [], [], 0.0, 0, 0
    for b0 in range(0, NIMG, BATCH):
        img = s["img"][b0:b0 + BATCH].cuda()
        ids, lens = eng.generate(img, early_stop=True)
        e2e_ids.append(ids.numpy().copy()); e2e_lens.append(lens.numpy().copy())
        if true_beam:
            continue
        # teacher forcing on the oracle's own captions, from the oracle's memory
        ref_ids, ref_lens = s["ids"][b0:b0 + BATCH], s["lens"][b0:b0 + BATCH]
        tok = np.concatenate([np.full((BATCH, 1), 2, np.int64), ref_ids[:, :T - 1]], axis=1)
        tok[tok == 0] = 4                                         # padding after an early stop: any valid id
        mem = s["mem"][b0:b0 + BATCH]
        lg = eng.decode_logits(mem.cuda(), torch.from_numpy(tok).int().cuda()).cpu()
        ref_lg, _ = O.transformer_logits(mem, torch.from_numpy(tok), s["Wv"], O.create_look_ahead_mask(T), T, num_layers=L)
        lp, lpr = torch.log_softmax(lg[..., :V], -1), torch.log_softmax(ref_lg, -1)
        lp_err = max(lp_err, float((lp - lpr).abs().max()))
        agree += int((lp.argmax(-1) == lpr.argmax(-1)).sum()); steps += lp.shape[0] * lp.shape[1]
        # ... and free-running decode from the oracle's memory (decoder-only sequence identity)
        ids, lens = eng.decode(early_stop=True)
        dec_ids.append(ids.numpy().copy()); dec_lens.append(lens.numpy().copy())
    eng.close()
    out = dict(e2e=(np.concatenate(e2e_ids), np.concatenate(e2e_lens)))
    if not true_beam:
        out.update(dec=(np.concatenate(dec_ids), np.concatenate(dec_lens)), lp_err=lp_err, agree=agree / steps)
    return out


def test_bf16x3_sequence_identity_99_percent(subject):
    s = subject
    r = _run(s, "bf16x3")
    same_e2e = _same(*r["e2e"], s["ids"], s["lens"]).mean()
    same_dec = _same(*r["dec"], s["ids"], s["lens"]).mean()
    _record("bf16x3", dict(images=NIMG, sequence_identity_e2e=float(same_e2e), sequence_identity_decoder_only=float(same_dec),
                           teacher_forced_logprob_max_abs_err=r["lp_err"], per_step_argmax_agreement=r["agree"]))
    print("bf16x3: identity e2e %.3f decoder-only %.3f, log-prob err %.2e, per-step agreement %.4f" % (same_e2e, same_dec, r["lp_err"], r["agree"]))
    assert r["lp_err"] < 2e-3
    assert same_dec >= 0.99 and same_e2e >= 0.99


def test_bf16x3_true_beam_sequence_identity(subject):
    s = subject
    r = _run(s, "bf16x3", true_beam=True)
    same = _same(*r["e2e"], s["ids_tb"], s["lens_tb"]).mean()
    _record("bf16x3_true_beam", dict(images=NIMG, sequence_identity_e2e=float(same)))
    assert same >= 0.99, same


def test_bf16_benchmarked_mode_parity_numbers(subject):
    s = subject
    r = _run(s, "bf16")
    same_e2e = _same(*r["e2e"], s["ids"], s["lens"]).mean()
    same_dec = _same(*r["dec"], s["ids"], s["lens"]).mean()
    # first step at which a caption leaves the oracle's, averaged (T = never)
    first = [int(np.argmax(a != b)) if (a != b).any() else T for a, b in zip(r["dec"][0], s["ids"])]
    _record("bf16", dict(images=NIMG, sequence_identity_e2e=float(same_e2e), sequence_identity_decoder_only=float(same_dec),
                         teacher_forced_logprob_max_abs_err=r["lp_err"], per_step_argmax_agreement=r["agree"],
                         mean_first_divergent_step_decoder_only=float(np.mean(first)), max_len=T))
    print("bf16: identity e2e %.3f decoder-only %.3f, log-prob err %.3f, per-step agreement %.4f" % (same_e2e, same_dec, r["lp_err"], r["agree"]))
    assert r["agree"] >= 0.95 and r["lp_err"] < 1.0, (r["agree"], r["lp_err"])
    assert same_dec >= 0.5, same_dec


def test_bf16_lanes_kernel_configuration_parity_numbers(subject):
    """The kernel set the bench's streamed figure runs on (fpnmt_config.lanes >= 2; forced here with opts tgemm_wide): wide-row
    Dense kernels (tgemmw_kernel), logits-free decode tail (softmax partials + 8 candidates per vocabulary tile merged by
    k_beam_step) and shared cache rows.  Same stated tolerance as the lanes = 1 configuration; both beam initialisations."""
    s = subject
    r = _run(s, "bf16", opts=("tgemm_wide",))
    same_e2e = _same(*r["e2e"], s["ids"], s["lens"]).mean()
    same_dec = _same(*r["dec"], s["ids"], s["lens"]).mean()
    rt = _run(s, "bf16", true_beam=True, opts=("tgemm_wide",))
    same_tb = _same(*rt["e2e"], s["ids_tb"], s["lens_tb"]).mean()
    _record("bf16_lanes_configuration", dict(images=NIMG, sequence_identity_e2e=float(same_e2e), sequence_identity_decoder_only=float(same_dec),
                                             teacher_forced_logprob_max_abs_err=r["lp_err"], per_step_argmax_agreement=r["agree"],
                                             true_beam_sequence_identity_e2e=float(same_tb)))
    print("bf16 (lanes configuration): identity e2e %.3f decoder-only %.3f true-beam e2e %.3f, log-prob err %.3f, per-step agreement %.4f"
          % (same_e2e, same_dec, same_tb, r["lp_err"], r["agree"]))
    assert r["agree"] >= 0.95 and r["lp_err"] < 1.0, (r["agree"], r["lp_err"])
    assert same_dec >= 0.5, same_dec


@pytest.mark.parametrize("true_beam,finished", [(False, False), (True, False), (True, True)])
def test_logits_free_tail_equals_logits_tail(subject, true_beam, finished):
    """Vocabulary projection + beam step with and without the [rows][V] logits tensor (opts no_vstats): the candidates are the
    same tokens; scores differ only by the summation order of the softmax denominator (per-tile partial sums), so nearly every
    caption must agree and the per-step scores to 5e-2 over whole captions.  The kernel-level bounds of the tail (the projection's
    partials and candidates, the beam step's merge, parents and tokens bit for bit) are in test_gpu_vocab_tail.py."""
    from fpnmt.engine import Engine
    s = subject
    res = []
    for opts in (("tgemm_wide",), ("tgemm_wide", "no_vstats")):
        eng = Engine(s["w"], backbone=BB, batch=BATCH, beam=N, vocab=V, max_len=T, num_layers=L, image_size=S, precision="bf16",
                     true_beam=true_beam, finished_beams=finished, length_penalty=0.6 if finished else 0.0, opts=opts)
        ids, lens, sc = eng.generate(s["img"][:BATCH].cuda(), early_stop=False, return_scores=True)
        ids_es, lens_es = eng.generate(s["img"][:BATCH].cuda(), early_stop=True)
        res.append((ids.clone(), lens.clone(), sc.cpu().clone(), ids_es.clone(), lens_es.clone()))
        eng.close()
    a, b = res
    same = (a[0] == b[0]).all(dim=1)
    assert same.float().mean() >= 0.95, same          # a flipped near-tie (scores within rounding) may move a caption
    assert torch.equal(a[1][same], b[1][same])
    fin = torch.isfinite(a[2]) & torch.isfinite(b[2])
    assert float((a[2][fin] - b[2][fin]).abs().max()) < 5e-2
    assert (a[3] == b[3]).all(dim=1).float().mean() >= 0.95
