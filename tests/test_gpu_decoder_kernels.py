"""GPU parity of the decoder's attention, cross-attention, KV-cache and input kernels, one at a time through the stand-alone
operators of the C ABI, against float64 references on the CPU.

Until these tests the decode kernels were seen only through whole-decoder logits (2e-2 rel-L2) and generated ids, bounds
at which a kernel that is wrong for one head, one step parity, positions >= 64, a chunk boundary, a padded memory token or
one member of a token-history class still passes.

Every reference is fed the values the kernel reads: activations rounded to bf16 or split into hi + lo (st_act), fp32 where
the engine uploads fp32 (embedding and positional tables, biases, LayerNorm parameters, the fp32 rows of layernorm_rows).
Bounds, from the kernels' arithmetic:
  * embed_pos, kv_reorder, the cache append of self-attention: bit-exact (one fp32 add, then st_act; copies).
  * layernorm_rows: the element-wise bound of tokens_ln_pos in test_gpu_encoder_kernels.py: rtol 2^-8 / 2^-15 (output
    rounding, bf16 / bf16x3) plus 2^-19 of |LN| + |gamma| |mean| / std (the fp32 mean, divided by the row's std).
  * attention (self and cross): |y - ref| <= rtol |ref| + eps * sum_j p_j |v_j|.  rtol is the output rounding.  eps is the
    relative error of the probabilities plus that of the fp32 P.V sum:
      - scores: q.k / 8 summed in fp32.  The CUDA-core kernels sum 8 products per lane and then 8 lanes by shuffles.  The
        mma.sync kernel sums 64 exact bf16 products in the tensor core's fp32 accumulator.  So the score error is at most
        n 2^-24 S with S = sum_i |q_i k_i| / 8 and n = 11 or 64, and a probability moves by twice that, relatively.
        __expf (ex2.approx of the rounded x log2 e) adds 2^-22 |s - m|.
      - P.V: Tk + 8 fp32 additions with the online-softmax rescales, (Tk + 8) 2^-24.
      - the mma.sync kernel feeds P to the tensor core as bf16 hi + lo: 2^-17 of p.
    So eps = 2 n 2^-24 max_j S_j + 2^-22 max_j |s_j - m| + (Tk + 8) 2^-24 [+ 2^-17], per (row, head).
  * xattn, three checks:
      1. The fold outputs Mt and Nt: one bf16 rounding (rtol 2^-8) of the fp64 fold of the bf16 inputs, plus the fp32
         accumulation of 64 products (64 2^-24 of sum |K| |Wq| / 8, or sum |Wo| |V|).  sbias: fp32 bq . K / 8, and exactly
         -1e30 at padded tokens.
      2. The output against the block recomputed in fp64 from the op's own Mt, Nt and sbias, with P rounded to bf16 as the
         kernel rounds it.  The kernel's fp32 probabilities can round to the other bf16 neighbour, so each LayerNorm input
         feature may move by 2^-8 p |Nt| for each such flip.  The scores are 32 k-steps of 16 products accumulated in
         fp32 (ds = 2^-19 max_hj sum_k |Mt| |x|, which moves p by 2 ds relatively), and the P.Nt sum adds 2^-20 of
         sum_hj p |Nt|.  The bound is (2 * 2^-8 max_hj p_hj |Nt[f, hj]| + (2^-20 + 2 ds) sum_hj p |Nt|) |gamma| / std,
         plus rtol 2^-8 |ref| and 2^-19 |gamma| |mean| / std.
      3. The output against the unfolded fp64 block LN(softmax((x Wq + bq) K^T / 8) V Wo + bo + x): rel-L2 per row
         <= 2e-2.  The fold rounds Mt and Nt to bf16 (2^-9 each, random over 512 and 128 terms) and P to bf16 (2^-9), which
         moves a row by a few 1e-3.  A wrong scale, a missing bias or a wrong operand index moves it by O(1).
Every output must be finite (outputs start as NaN), and whatever the kernel must not write (the other rows of out2, cache
positions other than the appended one) comes back bit for bit.

Self-attention inputs are built so that a read through the wrong row, parity or buffer pair cannot go unnoticed.  Every
cache entry that the active lineage does not read is NaN: position t of every row, the positions of rows no lineage
points at, and in the physical mode the whole unused buffer pair.  The inactive parity's table points at rows the active
one does not read at that position.  All indices stay in range; the poison is a value, never an address.

FPNMT_KERNEL_ERRORS=<path> merges the worst error of each operator, as a fraction of its bound, into that JSON file.

Measured on one B200 (1000 W power limit), worst error as a fraction of the bound, bf16 / bf16x3:
  self-attention mma.sync 0.95 / -, CUDA core 0.99 / 0.14 (split);  cross-attention 0.98 / 0.13;  layernorm_rows
  1.00 / 0.23;  embed_pos, kv_reorder and the cache append 0 mismatches;  xattn: fold Mt 0.99, Nt 0.99, sbias 0.06, block
  0.83, unfolded rel-L2 3.9e-3 against 2e-2.
In bf16 the output rounding alone reaches 2^-8 |y| at the bottom of a binade, so ratios near 1 there are that rounding.
The file runs in about 30 s.
"""
import numpy as np
import pytest
import torch

from kernel_check import RTOL, check_elementwise, error_report, gen, q_act, record  # noqa: F401 (error_report: autouse fixture)

pytestmark = pytest.mark.gpu

SENTINEL = -3.5
NAN = float("nan")


def same_bits(a, b):
    """Bit-pattern equality of fp32 tensors that treats every NaN alike."""
    return (a == b) | (torch.isnan(a) & torch.isnan(b))


# ------------------------------------------------------------------------------------------------------------------------
# decode self-attention
SA_MODES = [("mma", "bf16"), ("simt", "bf16"), ("split", "bf16x3")]
SA_KERNEL = {"mma": "mma", "simt": "simt", "split": "auto"}


def _partition(n, rng):
    """Random partition of beams 0..n-1 into classes, from all singletons to one class: rep[i] = first member."""
    labels = rng.integers(0, rng.integers(1, n + 1), n)
    first = {}
    return [first.setdefault(lab, i) for i, lab in enumerate(labels.tolist())]


def sa_inputs(rows, N, T, t, heads, physical, classes, prec, seed):
    """qkv, the cache pairs, anc (2, rows, T) and rep (2, rows) or None, following the engine's contract: the beams of image
    b are rows b*N .. b*N+N-1 (a trailing partial image when N does not divide rows); members of a token-history class share
    the representative's lineage and new K/V (never their queries)."""
    g, rng = gen(seed), np.random.default_rng(seed)
    d = heads * 64
    img = [np.arange(b, min(b + N, rows)) for b in range(0, rows, N)]
    par = t & 1
    # representatives per parity (identity without classes); the two parities get independent partitions
    rep = np.tile(np.arange(rows, dtype=np.int32), (2, 1))
    if classes:
        for p in range(2):
            for beams in img:
                rep[p, beams] = beams[_partition(len(beams), rng)]
    # lineage: at each position the image's rows read from a random half of its rows, the other parity from the rest
    anc = np.zeros((2, rows, T), np.int32)
    for beams in img:
        n = len(beams)
        for pos in range(T):
            perm = beams[rng.permutation(n)]
            k = max(1, n // 2)
            other = perm[k:] if n > 1 else np.array([(beams[0] + 1) % rows])   # one-row image: another image's row
            anc[par, beams, pos] = rng.choice(perm[:k], n)
            anc[1 - par, beams, pos] = rng.choice(other, n)
    anc[par] = anc[par, rep[par]]                               # members read their representative's lineage
    # queries along a per-(image, head) direction u; the key at position t-1 is 1.2 u (the maximum, in the last chunk)
    # and the other keys N(0, 4): scores span ~30
    u = torch.randn(len(img), heads, 64, generator=g)
    rimg = torch.arange(rows) // N
    qkv = torch.randn(rows, 3, heads, 64, generator=g)
    qkv[:, 0] = 2 * u[rimg] + 0.5 * qkv[:, 0]
    qkv[:, 1] *= 2
    qkv[:, 1:] = qkv[torch.from_numpy(rep[par].astype(np.int64)), 1:]      # members append the representative's K/V
    qkv = qkv.reshape(rows, 3 * d)
    kc = q_act(torch.randn(rows, T, heads, 64, generator=g) * 2, prec)
    vc = q_act(torch.randn(rows, T, heads, 64, generator=g), prec)
    if t >= 1:
        kc[:, t - 1] = q_act(1.2 * u[rimg], prec)
    read = torch.zeros(rows, T, dtype=torch.bool)
    read[torch.from_numpy(anc[par, :, :t].astype(np.int64)), torch.arange(t)] = True
    kc[~read], vc[~read] = NAN, NAN
    kc, vc = kc.reshape(rows * T, d), vc.reshape(rows * T, d)
    full_nan = torch.full((rows * T, d), NAN)
    if physical and par:                                        # odd steps live in the second pair
        pairs = [full_nan.clone(), full_nan.clone(), kc, vc]
    elif physical:
        pairs = [kc, vc, full_nan.clone(), full_nan.clone()]
    else:
        pairs = [kc, vc, None, None]
    return qkv, pairs, anc, (rep if classes else None)


def sa_reference(qkv, kc, vc, anc, t, T, heads, prec):
    """fp64 attention of every row over its lineage's cache entries and its own new position; also sum_j p_j |v_j|, the
    per-(row, head) score magnitude max_j sum_i |q_i k_ji| / 8 and spread max_j |s_j - m|."""
    rows, d = qkv.shape[0], heads * 64
    x = q_act(qkv, prec).double().reshape(rows, 3, heads, 64)
    q, kn, vn = x[:, 0], x[:, 1], x[:, 2]
    idx = torch.from_numpy(anc[t & 1, :, :t].astype(np.int64)) * T + torch.arange(t)
    K = torch.cat([kc.double()[idx].reshape(rows, t, heads, 64), kn.unsqueeze(1)], 1)
    V = torch.cat([vc.double()[idx].reshape(rows, t, heads, 64), vn.unsqueeze(1)], 1)
    s = torch.einsum("rhd,rjhd->rhj", q, K) / 8
    S = torch.einsum("rhd,rjhd->rhj", q.abs(), K.abs()) / 8
    p = torch.softmax(s, -1)
    ref = torch.einsum("rhj,rjhd->rhd", p, V)
    pv = torch.einsum("rhj,rjhd->rhd", p, V.abs())
    spread = (s.max(-1).values - s.min(-1).values)
    return ref.reshape(rows, d), pv, S.max(-1).values, spread


def sa_check(mode, prec, rows, N, T, t, heads, physical, classes, seed):
    from fpnmt.engine import dec_self_attention
    qkv, pairs, anc, rep = sa_inputs(rows, N, T, t, heads, physical, classes, prec, seed)
    before = [None if c is None else c.clone() for c in pairs]
    dev = [None if c is None else c.cuda() for c in pairs]
    y = dec_self_attention(qkv.cuda(), dev[0], dev[1], anc, t, heads, N, rep, dev[2], dev[3], SA_KERNEL[mode],
                           torch.full((rows, heads * 64), NAN).cuda(), prec).cpu()
    after = [None if c is None else c.cpu() for c in dev]
    # the append: exactly [row][t] of the active pair changes, to the row's stored K / V
    act = 2 if (physical and t & 1) else 0
    d = heads * 64
    new = q_act(qkv, prec).reshape(rows, 3, d)
    at = torch.arange(rows) * T + t
    for i, c in enumerate(after):
        if c is None:
            continue
        exp = before[i].clone()
        if i in (act, act + 1):
            exp[at] = new[:, 1 + i - act]
        bad = int((~same_bits(c, exp)).sum())
        record("dec_self_attention_append (mismatches)", bad, 1)
        assert bad == 0, "cache %d: %d elements differ from the expected append (only [row][t] of the active pair may change)" % (i, bad)
    kc, vc = before[act], before[act + 1]
    ref, pv, smax, spread = sa_reference(qkv, kc, vc, anc, t, T, heads, prec)
    n = 64 if mode == "mma" else 11
    eps = 2 * n * 2.0 ** -24 * smax + 2.0 ** -22 * spread + (t + 9) * 2.0 ** -24 + (2.0 ** -17 if mode == "mma" else 0.0)
    scale = (pv * eps.unsqueeze(-1)).reshape(rows, d)
    check_elementwise("dec_self_attention_%s/%s" % (mode, prec), y, ref, scale, RTOL[prec], 1.0)


T_SWEEP = [(T, t) for T in (8, 40, 72, 129) for t in (0, 1, 31, 32, 33, 63, 64, 65, T - 1) if t < T]
T_SWEEP = sorted(set(T_SWEEP))
PHYS_SWEEP = [(T, t) for (T, t) in T_SWEEP if t in (1, 32, 33, 64, 65, T - 1)]


@pytest.mark.parametrize("mode,prec", SA_MODES, ids=[m[0] for m in SA_MODES])
@pytest.mark.parametrize("T,t", T_SWEEP, ids=["T%d_t%d" % c for c in T_SWEEP])
def test_dec_self_attention_steps(T, t, mode, prec):
    sa_check(mode, prec, 6, 3, T, t, 8, False, False, T * 1000 + t)


@pytest.mark.parametrize("mode,prec", SA_MODES, ids=[m[0] for m in SA_MODES])
@pytest.mark.parametrize("T,t", PHYS_SWEEP, ids=["T%d_t%d" % c for c in PHYS_SWEEP])
def test_dec_self_attention_physical(T, t, mode, prec):
    sa_check(mode, prec, 6, 3, T, t, 8, True, False, T * 1000 + t + 7)


SHAPES = [
    # name, rows, N, T, t, heads, physical
    ("h1_rows9", 9, 3, 40, 35, 1, False),             # 9 warps: not a multiple of 4 or 14
    ("h3_rows5", 5, 5, 72, 66, 3, True),              # 15 warps
    ("h3_rows7_beam1", 7, 1, 40, 33, 3, False),       # one row per image
    ("h8_rows640_wave", 640, 8, 72, 40, 8, False),    # 5120 warps: more than one wave of either kernel
]


@pytest.mark.parametrize("mode,prec", SA_MODES, ids=[m[0] for m in SA_MODES])
@pytest.mark.parametrize("case", SHAPES, ids=[c[0] for c in SHAPES])
def test_dec_self_attention_shapes(case, mode, prec):
    name, rows, N, T, t, heads, physical = case
    sa_check(mode, prec, rows, N, T, t, heads, physical, False, len(name) * 13 + rows)


CLASS_CASES = [
    # name, rows, N, T, t, physical
    ("n2_t0", 8, 2, 40, 0, False),
    ("n4_t5", 12, 4, 40, 5, True),
    ("n8_t33", 24, 8, 72, 33, False),
    ("n8_t70", 16, 8, 72, 70, True),
    ("n8_t64_wave", 640, 8, 72, 64, False),
    ("n9_rep_ignored", 18, 9, 40, 21, False),
    ("n16_rep_ignored", 32, 16, 72, 66, True),
    ("rows10_n4_rep", 10, 4, 40, 31, False),          # N does not divide rows: every row is its own class
    ("rows7_n2_rep", 7, 2, 72, 65, True),
]


@pytest.mark.parametrize("mode,prec", SA_MODES, ids=[m[0] for m in SA_MODES])
@pytest.mark.parametrize("case", CLASS_CASES, ids=[c[0] for c in CLASS_CASES])
def test_dec_self_attention_classes(case, mode, prec):
    name, rows, N, T, t, physical = case
    sa_check(mode, prec, rows, N, T, t, 8, physical, True, len(name) * 17 + rows + t)


# ------------------------------------------------------------------------------------------------------------------------
# decode cross-attention (CUDA-core kernel): K / V of the last layer of an L*1024-wide memory projection, other columns NaN
CA_TK = [1, 4, 16, 31, 32, 33, 64, 100]
CA_BEAM = [1, 3, 16]


@pytest.mark.parametrize("prec", ["bf16", "bf16x3"])
@pytest.mark.parametrize("beam", CA_BEAM)
@pytest.mark.parametrize("tk", CA_TK)
def test_dec_cross_attention(tk, beam, prec):
    from fpnmt.engine import dec_cross_attention
    B, heads, L = 3, 8, 3
    kv_ld, k_col, v_col = L * 1024, (L - 1) * 1024, (L - 1) * 1024 + 512
    g = gen(tk * 100 + beam)
    u = torch.randn(B, heads, 64, generator=g)
    q = (2 * u.repeat_interleave(beam, 0) + 0.5 * torch.randn(B * beam, heads, 64, generator=g)).reshape(B * beam, 512)
    k = torch.randn(B, tk, heads, 64, generator=g) * 2
    k[:, -1] = 1.2 * u
    kv = torch.full((B, tk, kv_ld), NAN)
    kv[..., k_col:k_col + 512] = k.reshape(B, tk, 512)
    kv[..., v_col:v_col + 512] = torch.randn(B, tk, 512, generator=g)
    kv = kv.reshape(B * tk, kv_ld)
    y = dec_cross_attention(q.cuda(), kv.cuda(), beam, heads, k_col, v_col, torch.full((B * beam, 512), NAN).cuda(), prec).cpu()
    qq = q_act(q, prec).double().reshape(B, beam, heads, 64)
    kq = q_act(kv, prec).double().reshape(B, tk, kv_ld)
    K = kq[..., k_col:k_col + 512].reshape(B, tk, heads, 64)
    V = kq[..., v_col:v_col + 512].reshape(B, tk, heads, 64)
    s = torch.einsum("bnhd,bjhd->bnhj", qq, K) / 8
    S = torch.einsum("bnhd,bjhd->bnhj", qq.abs(), K.abs()).max(-1).values / 8
    p = torch.softmax(s, -1)
    ref = torch.einsum("bnhj,bjhd->bnhd", p, V)
    pv = torch.einsum("bnhj,bjhd->bnhd", p, V.abs())
    eps = 2 * 11 * 2.0 ** -24 * S + 2.0 ** -22 * (s.max(-1).values - s.min(-1).values) + (tk + 8) * 2.0 ** -24
    check_elementwise("dec_cross_attention/" + prec, y.reshape(B, beam, heads, 64), ref, pv * eps.unsqueeze(-1), RTOL[prec], 1.0)


# ------------------------------------------------------------------------------------------------------------------------
# fused cross-attention block (bf16): fold kernels + one tcgen05 kernel per image of the slice
def bf(x):
    return x.to(torch.bfloat16).double()


def xa_inputs(Btot, n_mem, L, beam, g, flat_images=()):
    """ckv (Btot*n_mem, L*1024); weights; out1 (Btot*beam, 512).  Images in flat_images get out1 rows of exactly 100 and V
    scaled so that the LayerNorm input has mean ~100 and std ~1e-2."""
    ckv = torch.randn(Btot, n_mem, L, 2, 512, generator=g)
    ckv[:, :, :, 0] *= 3                                        # K: scores of std ~3
    wq = (torch.randn(L, 512, 512, generator=g) / 512 ** 0.5).numpy()
    bq = (torch.randn(L, 512, generator=g) * 0.5).numpy()
    wo = (torch.randn(L, 512, 512, generator=g) / 512 ** 0.5).numpy()
    bo = (torch.randn(512, generator=g) * (1e-2 if flat_images else 0.5)).numpy()
    gamma = (torch.rand(512, generator=g) + 0.5).numpy()
    beta = (torch.randn(512, generator=g) * 0.1).numpy()
    out1 = torch.randn(Btot, beam, 512, generator=g)
    for b in flat_images:
        out1[b] = 100.0
        ckv[b, :, :, 1] *= 1e-2
    return ckv.reshape(Btot * n_mem, L * 1024), wq, bq, wo, bo, gamma, beta, out1.reshape(Btot * beam, 512)


def ln64(x, gamma, beta):
    mean = x.mean(-1, keepdim=True)
    var = ((x - mean) ** 2).mean(-1, keepdim=True)
    std = torch.sqrt(var + 1e-6)
    return (x - mean) / std * gamma + beta, mean, std


XA_CASES = [
    # name, beam, n_mem, Btot, b0, B, layer, flat images
    ("beam1_nm16_l0", 1, 16, 4, 0, 4, 0, ()),
    ("beam3_nm4_l2_slice", 3, 4, 5, 2, 3, 2, ()),
    ("beam8_nm16_l0_slice", 8, 16, 6, 1, 4, 0, (2,)),
    ("beam15_nm15_l2_slice", 15, 15, 3, 1, 1, 2, ()),
    ("beam16_nm1_l2", 16, 1, 3, 0, 3, 2, (1,)),
    ("beam16_nm16_l0_slice", 16, 16, 4, 3, 1, 0, ()),
    ("beam8_nm16_b300_l2", 8, 16, 302, 2, 300, 2, (5, 150)),
]


@pytest.mark.parametrize("case", XA_CASES, ids=[c[0] for c in XA_CASES])
def test_xattn(case):
    from fpnmt.engine import xattn
    name, beam, n_mem, Btot, b0, B, layer, flat = case
    L = 3
    g = gen(len(name) * 7 + Btot)
    ckv, wq, bq, wo, bo, gamma, beta, out1 = xa_inputs(Btot, n_mem, L, beam, g, flat)
    out2 = torch.full((Btot * beam, 512), SENTINEL)
    out2[b0 * beam:(b0 + B) * beam] = NAN
    y, mt, nt, sb = xattn(ckv.cuda(), wq, bq, wo, bo, gamma, beta, out1.cuda(), beam, layer, b0, B, out2.cuda(), True)
    y, mt, nt, sb = y.cpu(), mt.cpu().double(), nt.cpu().double(), sb.cpu().double()
    outside = torch.ones(Btot * beam, dtype=torch.bool)
    outside[b0 * beam:(b0 + B) * beam] = False
    assert bool((y[outside] == SENTINEL).all()), "xattn wrote rows outside the images [b0, b0 + B)"
    y = y[~outside].double().reshape(B, beam, 512)

    # ---- 1. the fold, for the images of the slice and the layer it runs
    kv = bf(ckv).reshape(Btot, n_mem, L, 2, 8, 64)[b0:b0 + B, :, layer]            # (B, j, 2, h, d)
    K, V = kv[:, :, 0], kv[:, :, 1]                                               # (B, j, h, d)
    Wq = bf(torch.from_numpy(wq[layer])).reshape(512, 8, 64)                      # [k][h][d]
    Wo = bf(torch.from_numpy(wo[layer])).reshape(8, 64, 512)                      # [h][d][f]
    bqd = torch.from_numpy(bq[layer]).double().reshape(8, 64)
    mt_ref = torch.einsum("bjhd,khd->bhjk", K, Wq) / 8
    mt_sc = torch.einsum("bjhd,khd->bhjk", K.abs(), Wq.abs()) / 8
    nt_ref = torch.einsum("bjhd,hdf->bfhj", V, Wo)
    nt_sc = torch.einsum("bjhd,hdf->bfhj", V.abs(), Wo.abs())
    sb_ref = torch.einsum("bjhd,hd->bhj", K, bqd) / 8
    sb_sc = torch.einsum("bjhd,hd->bhj", K.abs(), bqd.abs()) / 8
    base = layer * Btot + b0
    mt_k = mt.reshape(L * Btot, 8, 16, 512)[base:base + B]
    nt_k = nt.reshape(L * Btot, 512, 8, 16)[base:base + B]
    sb_k = sb.reshape(L * Btot, 8, 16)[base:base + B]
    assert bool((sb_k[:, :, n_mem:] == float(np.float32(-1e30))).all()), "sbias must be exactly -1e30 at the padded memory tokens"
    check_elementwise("xattn_fold_Mt", mt_k[:, :, :n_mem], mt_ref, mt_sc, RTOL["bf16"], 64 * 2.0 ** -24)
    check_elementwise("xattn_fold_Nt", nt_k[..., :n_mem], nt_ref, nt_sc, RTOL["bf16"], 64 * 2.0 ** -24)
    check_elementwise("xattn_fold_sbias", sb_k[:, :, :n_mem], sb_ref, sb_sc, 2.0 ** -22, 64 * 2.0 ** -24)

    x = bf(out1).reshape(Btot, beam, 512)[b0:b0 + B]                              # (B, n, k)
    bod, gd, betad = (torch.from_numpy(a).double() for a in (bo, gamma, beta))

    # ---- 2. the block from the op's own Mt / Nt / sbias, P rounded to bf16
    s = torch.einsum("bhjk,bnk->bnhj", mt_k, x) + sb_k.unsqueeze(1)               # (B, n, h, 16) with the padding
    p = torch.softmax(s, -1)
    pb = bf(p)
    xin = torch.einsum("bfhj,bnhj->bnf", nt_k, pb) + bod + x
    ref2, mean2, std2 = ln64(xin, gd, betad)
    flips = torch.cat([(nt_k[i:i + 8].abs().flatten(-2).unsqueeze(1) * p[i:i + 8].flatten(-2).unsqueeze(2)).amax(-1)
                       for i in range(0, B, 8)])
    ds = 2.0 ** -19 * torch.einsum("bhjk,bnk->bnhj", mt_k.abs(), x.abs()).flatten(-2).amax(-1, keepdim=True)
    pnt = torch.einsum("bfhj,bnhj->bnf", nt_k.abs(), p)
    scale = gd.abs() / std2 * (2 * 2.0 ** -8 * flips + (2.0 ** -20 + 2 * ds) * pnt + 2.0 ** -19 * mean2.abs())
    check_elementwise("xattn_block", y, ref2, scale, RTOL["bf16"], 1.0)

    # ---- 3. the unfolded block in fp64
    q2 = torch.einsum("bnk,khd->bnhd", x, Wq) + bqd
    s3 = torch.einsum("bnhd,bjhd->bnhj", q2, K) / 8
    att = torch.einsum("bnhj,bjhd->bnhd", torch.softmax(s3, -1), V)
    ref3, _, _ = ln64(torch.einsum("bnhd,hdf->bnf", att, Wo) + bod + x, gd, betad)
    rel = (y - ref3).norm(dim=-1) / ref3.norm(dim=-1)
    worst = float(rel.max())
    record("xattn_unfolded (rel-L2 per row)", worst, 2e-2)
    assert worst <= 2e-2, "%s: a row is %.3g rel-L2 from the unfolded block (row %s)" % (name, worst, divmod(int(rel.argmax()), beam))


# ------------------------------------------------------------------------------------------------------------------------
# physical KV-cache reorder: 16-byte units, 4 x 256 per main-loop iteration.  D = 512: a position is 64 units in bf16 and 128
# (hi + lo) in bf16x3, so t = 16 / 8 ends exactly on the main loop and t = 17 / 9 one position past it.
KV_CASES = [("bf16", t) for t in (0, 1, 15, 16, 17, 40)] + [("bf16x3", t) for t in (0, 1, 8, 9, 40)]


@pytest.mark.parametrize("prec,t", KV_CASES, ids=["%s_t%d" % c for c in KV_CASES])
def test_kv_reorder(prec, t):
    from fpnmt.engine import kv_reorder
    nc, B, N, T, D = 3, 3, 4, 40, 512
    rows = B * N
    g = gen(t * 10 + len(prec))
    src = q_act(torch.randn(nc, rows, T, D, generator=g), prec)
    dst = q_act(torch.randn(nc, rows, T, D, generator=g) + 10, prec)
    parent = np.zeros((T, rows), np.int32)
    for tt in range(T):                      # image 0 repeats parents, image 1 permutes them, image 2 mixes
        parent[tt, 0:N] = torch.randint(0, N, (N,), generator=g).numpy()
        parent[tt, N:2 * N] = torch.randperm(N, generator=g).numpy()
        parent[tt, 2 * N:] = [N - 1, N - 1, 0, 1]
    y = kv_reorder(src.cuda(), dst.clone().cuda(), parent, N, t, prec).cpu()
    exp = dst.clone()
    if t > 0:
        srow = (torch.arange(rows) // N) * N + torch.from_numpy(parent[t - 1].astype(np.int64))
        exp[:, :, :t] = src[:, srow, :t]
    bad = int((~same_bits(y, exp)).sum())
    record("kv_reorder/%s (mismatches)" % prec, bad, 1)
    assert bad == 0, "t = %d: %d cache elements differ from the reordered copy" % (t, bad)


# ------------------------------------------------------------------------------------------------------------------------
# decoder input: one thread per 8 channels of a row
EMB_CASES = [("c512", 12, 512, 11), ("c24_ragged", 37, 24, 11), ("c512_t0", 5, 512, 0)]


@pytest.mark.parametrize("prec", ["bf16", "bf16x3"])
@pytest.mark.parametrize("case", EMB_CASES, ids=[c[0] for c in EMB_CASES])
def test_embed_pos(case, prec):
    from fpnmt.engine import embed_pos
    name, rows, C, t = case
    V, T = 50, 12
    g = gen(rows * 3 + C)
    emb = torch.randn(V, C, generator=g) * 3
    pos = torch.randn(T, C, generator=g)
    tok = torch.randint(0, V, (rows,), generator=g)
    tok[0], tok[-1] = 0, V - 1
    y = embed_pos(tok.numpy(), emb.numpy(), pos.numpy(), t, torch.full((rows, C), NAN).cuda(), prec).cpu()
    exp = q_act(emb[tok] + pos[t], prec)
    bad = int((y != exp).sum())
    record("embed_pos/%s (mismatches)" % prec, bad, 1)
    assert bad == 0, "%s: %d outputs differ from emb[tok] + pos[t]" % (name, bad)


# ------------------------------------------------------------------------------------------------------------------------
# LayerNorm of fp32 rows (the unfused decoder): one warp per 512-wide row, 8 rows per block
@pytest.mark.parametrize("prec", ["bf16", "bf16x3"])
@pytest.mark.parametrize("rows", [1, 7, 13, 100])
def test_layernorm_rows(rows, prec):
    from fpnmt.engine import layernorm_rows
    g = gen(rows * 5)
    x = torch.randn(rows, 512, generator=g) * 2 + 0.5
    x[::3] = 100 + torch.randn(x[::3].shape, generator=g) * 1e-2
    x[1::4] = 3.7                                              # constant rows: LN = beta
    gamma = (torch.rand(512, generator=g) + 0.5).numpy()
    beta = (torch.randn(512, generator=g) * 0.1).numpy()
    y = layernorm_rows(x.cuda(), gamma, beta, 1e-6, torch.full((rows, 512), NAN).cuda(), prec).cpu()
    xd = x.double()
    gd, bd = torch.from_numpy(gamma).double(), torch.from_numpy(beta).double()
    ref, mean, std = ln64(xd, gd, bd)
    scale = ref.abs() + gd.abs() * mean.abs() / std
    check_elementwise("layernorm_rows/" + prec, y, ref, scale, RTOL[prec], 2.0 ** -19)


# ------------------------------------------------------------------------------------------------------------------------
# argument checks: out-of-range tables and unsupported shapes are rejected before anything reaches the device
def _rejects(fn):
    from fpnmt._lib import ERR_INVALID, FpnmtError
    with pytest.raises(FpnmtError) as e:
        fn()
    assert e.value.code == ERR_INVALID


def test_decoder_ops_reject_bad_arguments():
    from fpnmt.engine import dec_self_attention, embed_pos, kv_reorder, xattn
    rows, T, d = 4, 8, 64
    qkv = torch.zeros(rows, 3 * d).cuda()
    cache = lambda: torch.zeros(rows * T, d).cuda()
    anc = np.zeros((2, rows, T), np.int32)
    bad = anc.copy()
    bad[1, 2, 7] = rows
    _rejects(lambda: dec_self_attention(qkv, cache(), cache(), bad, 3, 1, 2))
    bad[1, 2, 7] = -1
    _rejects(lambda: dec_self_attention(qkv, cache(), cache(), bad, 3, 1, 2))
    _rejects(lambda: dec_self_attention(qkv, cache(), cache(), anc, 3, 1, 2, np.full((2, rows), rows)))
    _rejects(lambda: dec_self_attention(qkv, cache(), cache(), anc, T, 1, 2))
    _rejects(lambda: dec_self_attention(qkv, cache(), cache(), anc, 3, 1, 2, kernel="mma", precision="bf16x3"))
    par = np.zeros((T, rows), np.int32)
    par[5, 3] = 2
    _rejects(lambda: kv_reorder(torch.zeros(1, rows, T, 512).cuda(), torch.zeros(1, rows, T, 512).cuda(), par, 2, 3))
    _rejects(lambda: embed_pos(np.array([0, 10]), np.zeros((10, 16), np.float32), np.zeros((4, 16), np.float32), 1))
    _rejects(lambda: embed_pos(np.array([0, 1]), np.zeros((10, 12), np.float32), np.zeros((4, 12), np.float32), 1))
    w = np.zeros((1, 512, 512), np.float32)
    v = np.zeros(512, np.float32)
    ckv17 = torch.zeros(17, 1024).cuda()
    _rejects(lambda: xattn(ckv17, w, v[None], w, v, v, v, torch.zeros(2, 512).cuda(), 2, 0))        # n_mem 17
    ckv = torch.zeros(4, 1024).cuda()
    _rejects(lambda: xattn(ckv, w, v[None], w, v, v, v, torch.zeros(17, 512).cuda(), 17, 0))        # beam 17
    _rejects(lambda: xattn(ckv, w, v[None], w, v, v, v, torch.zeros(2, 512).cuda(), 2, 0, precision="bf16x3"))
