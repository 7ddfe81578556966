"""KV-cache modes of the per-operator decode chain (north-star item 3, SURVEY 8d):
  ancestry : the cache never moves; a per-beam ancestry table maps (beam, position) to the physical row (default)
  physical : after every step ONE bandwidth kernel (k_kv_reorder) gathers the live span of every cache row of all layers from
             its beam parent's row into the other buffer pair; attention then reads its own row.
Both read exactly the same K/V values with the same kernels, so ids, lengths, per-step scores and teacher-forced logits must
be BIT-IDENTICAL - with the reference's beam initialisation (parent = identity) and with true beams (real permutations)."""
import pytest
import torch

import fpnmt_oracle as O

pytestmark = pytest.mark.gpu

BB, S, L, V, T, N, B = "mobilenet224_1.0", 256, 2, 1000, 12, 8, 6


@pytest.mark.parametrize("prec", ["bf16", "bf16x3"])
@pytest.mark.parametrize("true_beam", [False, True])
def test_physical_reorder_equals_ancestry_table(prec, true_beam):
    from fpnmt.engine import Engine
    w = O.caption_weights(BB, vocab=V, layers=L, seed=0, end_bias=6.0)
    img = O.test_images(B, S, seed=41).cuda()
    gtok = torch.randint(4, V, (B, T), generator=torch.Generator().manual_seed(2))
    gtok[:, 0] = 2
    res = {}
    for mode in ("ancestry", "physical"):
        eng = Engine(w, backbone=BB, batch=B, beam=N, vocab=V, max_len=T, num_layers=L, image_size=S, precision=prec,
                     true_beam=true_beam, cache_mode=mode, decode_path="chain")
        ids, lens, sc = eng.generate(img, early_stop=False, return_scores=True)
        ids_es, lens_es = eng.generate(img, early_stop=True)
        lg = eng.decode_logits(None, gtok.int().cuda()).cpu()
        ids_again, _ = eng.generate(img, early_stop=False)            # the forced run must not disturb a later decode
        assert torch.equal(ids, ids_again)
        res[mode] = (ids.clone(), lens.clone(), sc.cpu().clone(), ids_es.clone(), lens_es.clone(), lg)
        eng.close()
    a, p = res["ancestry"], res["physical"]
    assert torch.equal(a[0], p[0]) and torch.equal(a[1], p[1])
    assert torch.equal(a[2], p[2])
    assert torch.equal(a[3], p[3]) and torch.equal(a[4], p[4])
    assert torch.equal(a[5], p[5])
    if true_beam:      # the permutations are real: the beams of at least one image have reordered
        assert len({tuple(r.tolist()) for r in a[0]}) > 1


def test_physical_mode_is_rejected_where_it_cannot_run():
    from fpnmt._lib import FpnmtError
    from fpnmt.engine import Engine
    w = O.caption_weights(BB, vocab=512, layers=L, seed=1)
    with pytest.raises(FpnmtError):
        Engine(w, backbone=BB, batch=2, beam=4, vocab=512, max_len=8, num_layers=L, image_size=S, cache_mode="physical", decode_path="fused")


@pytest.mark.parametrize("true_beam,finished", [(False, False), (True, False), (True, True)])
def test_shared_cache_rows_of_identical_beams_change_nothing(true_beam, finished):
    """Ancestry mode points a beam at the cache rows of the first beam of its image with the same token history
    (BeamState::rep); with the sharing switched off (opts no_kv_share) every beam walks its own lineage.  Same bits either way:
    ids, lengths and per-step scores are identical, under the reference's identical beams and under true beams."""
    from fpnmt.engine import Engine
    w = O.caption_weights(BB, vocab=V, layers=L, seed=3, end_bias=6.0)
    img = O.test_images(B, S, seed=43).cuda()
    res = []
    for opts in ((), ("no_kv_share",)):
        eng = Engine(w, backbone=BB, batch=B, beam=N, vocab=V, max_len=T, num_layers=L, image_size=S, precision="bf16",
                     true_beam=true_beam, finished_beams=finished, length_penalty=0.6 if finished else 0.0, decode_path="chain", opts=opts)
        ids, lens, sc = eng.generate(img, early_stop=False, return_scores=True)
        ids_es, lens_es = eng.generate(img, early_stop=True)
        res.append((ids.clone(), lens.clone(), sc.cpu().clone(), ids_es.clone(), lens_es.clone()))
        eng.close()
    for x, y in zip(*res):
        assert torch.equal(x, y)
