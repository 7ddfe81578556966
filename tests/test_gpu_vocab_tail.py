"""GPU parity of the logits-free decode tail, one kernel at a time: the vocabulary projection in its softmax-partials epilogue
(tgemmw_kernel with TgemmParams::vs_*, through fpnmt_op_vocab_stats) and the beam step's merge of those partials (k_beam_step's
vs_stat branch, through fpnmt_beam_step_vstats), against float64 references and the CPU oracle.

The beam-search decode of the bf16 mode with the wide Dense kernels (every lane configuration, so the default benchmark) never
writes the [rows][V] logits: per (row, 128-feature tile) the projection leaves (max, sum exp(z - max)) and the tile's 8 largest
logits with their ids, and the beam step folds them into the row's log-sum-exp and top N.  Until these tests the tail was
seen only through whole captions (95 % identical captions, step scores within 5e-2), bounds at which a tile left out of the
log-sum-exp, ids off by one tile, a flipped tie order, padding features taken as tokens or a wrong row slot still pass.

Bounds (u = 2^-24; every bound is derived from the kernels' arithmetic, none is fitted):
  * Projection, exact inputs: x = a/8 and W = b/16 with small integers a, b (exact in bf16), bias a multiple of 1/128.  Every
    logit is then an fp32 number whatever the accumulation order (|z| 128 < 2^17, far below 2^24), so the tile maximum, the 8
    candidate values, their ids (ties: lower id first, the tf.math.top_k order) and the -inf / 0x7fffffff padding are compared
    bit for bit.
  * sum exp(z - max) of a tile: the epilogue walks 4 chunks of 32 features with an online maximum.  A term passes through at
    most 4 __expf calls (its own and up to 3 rescales of the running sum), each ex2.approx (relative error <= 2^-22) of an
    argument rounded twice (x - m and the product with log2 e, and the rounded constant): 2^-22 + 3 u D <= 2^-22 (1 + D) with
    D = max - z >= every rescale argument of the term.  The sum itself is 4 x (31 adds + 1 multiply + 1 add) <= 136 fp32
    roundings, each at most u of a partial sum that the later rescales keep below the final sum S.  So
        |S_gpu - S| <= 136 u S + sum_i exp(-D_i) 2^-20 (1 + D_i)   (+ 2^-119 for flushed subnormal terms).
  * Projection, random inputs: the reference is fp64 of the bf16-rounded x and W and the fp32 bias.  The tensor core's fp32
    accumulation of K exact bf16 products may be off by one unit in the last place per addition (truncation included), and the
    bias add rounds once: delta = K 2^-23 sum_k |x_k w_k| + u |z|.  Maxima and candidate values within delta (the k-th largest
    of values each moved by <= delta moves by <= delta); ids only where the fp64 gap to both neighbouring ranks exceeds
    2 delta; sum exp within the bound above plus S (exp(2 delta) - 1).
  * Merge (log scores): the beam step folds the tiles' (m_t, S_t) with two __expf rescales per tile (thread -> warp,
    warp -> block), a 5-step warp sum and an 8-term block sum (15 roundings of the total); then lse = m + logf(sum) (logf <= 1
    ulp, the add u |lse|), and a candidate's score is score + (z - lse) (two more roundings).  With w_t = S_t exp(m_t - m):
        eps_sum = 15 u + sum_t w_t (e_t + 2^-21 (1 + m - m_t)) / sum_t w_t
        |score_gpu - score_fp64| <= eps_sum (1 + 1e-3) + 2^-23 |log sum| + u |lse| + u |z - lse| + u |score + z - lse|
    where e_t is the relative error of S_t: u for partials rounded from fp64 on the host, the projection's bound above when
    they come from the kernel (composition).  The logits path (k_beam_step on [rows][V] fp32) has 3 __expf per element and
    4 nv4 + 23 roundings of its sum (nv4 float4 slots per thread), the same formula otherwise; the two paths' scores agree
    within the sum of their bounds.
Parents and tokens are compared bit for bit with fpnmt_oracle.beam_step and with the logits path on the same logits.

Planted cases: all top-8 of a row in one tile; one winner per tile; the row maximum at the last valid feature of the last
tile; equal logits at features 127 / 128 and inside one tile; a row whose logits are all equal (x = 0, no bias); rows >= R of
the outputs poisoned (NaN, sentinel ids) must come back bit for bit.  Merge trials: random, identical rows (the reference's
start state), ties across a tile boundary, all top N in one tile, peaked rows, dead beams (score -inf, the true-beam start
state), and fewer valid tokens than beams (host-built partials of a vocabulary smaller than N, so the cnt < N padding runs
right after a call that left real candidates in the engine's candidate buffers).

FPNMT_KERNEL_ERRORS=<path> merges the worst error of each check, as a fraction of its bound, into that JSON file.

Measured on one B200 (1000 W power limit), worst error as a fraction of the bound:
  projection, exact inputs: tile maxima, candidate values, ids and padding 0 mismatches, sum exp 0.057;  random inputs: maxima
  and candidate values 0.0043, sum exp 0.020;  merge score against fp64 0.49, the logits path 0.43, the two paths against
  each other 0.18 (of the sum of their bounds);  projection -> merge 0.034;  parents and tokens 0 mismatches.
The ratios near 0.5 are the final fp32 rounding of the score itself (u |score|); the sum-exp bounds carry the worst-case
4 __expf errors per term, which random data does not reach.  The file runs in about 17 s.
"""
import zlib

import numpy as np
import pytest
import torch

import fpnmt_oracle as O
from kernel_check import error_report, gen, q_act, record  # noqa: F401 (error_report: autouse fixture)

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
TILE, NC = 128, 8
PAD_ID = 0x7FFFFFFF
SENTINEL_ID = -7


# ------------------------------------------------------------------------------------------------------------------------
# fp64 references
def tile_reference(z, F):
    """Per (row, 128-feature tile) of fp64 logits z (R, F): max, sum exp(z - max), the 8 largest (ties: lower id first) with
    their ids (-inf / 0x7fffffff padded), and the terms exp(-D), D = max - z, of the sum (0 at padding)."""
    R = z.shape[0]
    ft = (F + TILE - 1) // TILE
    zp = np.full((R, ft * TILE), -np.inf)
    zp[:, :F] = z
    zt = zp.reshape(R, ft, TILE)
    m = zt.max(-1)
    D = m[..., None] - zt
    t = np.exp(-D)
    S = t.sum(-1)
    order = np.argsort(-zt, axis=-1, kind="stable")[..., :NC]
    val = np.take_along_axis(zt, order, -1)
    ids = order + (np.arange(ft) * TILE)[None, :, None]
    ids = np.where(val == -np.inf, PAD_ID, ids)
    return m, S, val, ids, t, np.where(np.isfinite(D), D, 0.0)


def sumexp_bound(S, t, D):
    """The projection's bound on sum exp(z - max) per (row, tile) (module docstring)."""
    return 136 * U * S + (t * 2.0 ** -20 * (1 + D)).sum(-1) + 2.0 ** -119


def host_partials(logits, F=None):
    """stat / val / idx exactly as the projection defines them, from fp32 logits (rows, >= F): fp32 tile maxima, the fp64
    sum exp rounded to fp32, the 8 largest logits and their ids."""
    F = logits.shape[1] if F is None else F
    m, S, val, ids, _, _ = tile_reference(logits[:, :F].double().numpy(), F)
    stat = np.stack([m, S], -1).astype(np.float32)
    return (torch.from_numpy(stat), torch.from_numpy(val.astype(np.float32)), torch.from_numpy(ids.astype(np.int32)))


def lse_terms(m_t, S_t, e_t):
    """(lse, eps_sum, log sum) of the vs_stat merge from the tiles' fp64 (max, sum exp) and S_t's relative error e_t."""
    m = m_t.max(-1, keepdims=True)
    w = S_t * np.exp(m_t - m)
    ws = w.sum(-1)
    eps = 15 * U + (w * (e_t + 2.0 ** -21 * (1 + m - m_t))).sum(-1) / ws
    return m[:, 0] + np.log(ws), eps, np.log(ws)


def merge_bound(lse, eps, logsum, z, score):
    return eps * (1 + 1e-3) + 2.0 ** -23 * np.abs(logsum) + U * np.abs(lse) + U * np.abs(z - lse) + U * np.abs(score + z - lse)


def logits_path_eps(z):
    """eps_sum of k_beam_step's logits path on fp64 logits z (rows, V)."""
    V = z.shape[1]
    threads = 256 if V <= 16384 else 512
    nv4 = (V + 4 * threads - 1) // (4 * threads)
    m = z.max(-1, keepdims=True)
    w = np.exp(z - m)
    return (4 * nv4 + 23) * U + (w * 3 * 2.0 ** -22 * (1 + m - z)).sum(-1) / w.sum(-1)


# ------------------------------------------------------------------------------------------------------------------------
# (a) the vocabulary projection: softmax partials and candidates
# name, R, K, F, exact inputs, bias, first planted pattern
PROJ_CASES = [
    ("R1_F1000", 1, 512, 1000, True, True, 2),
    ("R40_F8_one_tile", 40, 512, 8, True, False, 0),
    ("R128_F1032_last_tile_8", 128, 512, 1032, True, True, 1),
    ("R129_K2048_F1000", 129, 2048, 1000, True, False, 3),
    ("R300_F10000", 300, 512, 10000, True, True, 4),
    ("R1024_F1032", 1024, 512, 1032, True, False, 0),
    ("R40_F24576_192_tiles", 40, 512, 24576, True, True, 1),
    ("random_R300_F1000", 300, 512, 1000, False, True, 0),
    ("random_R129_K2048_F1032", 129, 2048, 1032, False, True, 2),
    ("random_R1024_F10000", 1024, 512, 10000, False, True, 3),
]
N_PATTERNS = 5


def plant(x, W, bias, F, rows, first):
    """Plants the five row patterns (in rotation from `first`) into rows `rows` through reserved input columns: row r_p reads
    only column p of x (x = 1), so its logits are W[p] + bias, and no other row reads column p."""
    x[:, :N_PATTERNS] = 0
    ft = (F + TILE - 1) // TILE
    for j, r in enumerate(rows):
        p = (first + j) % N_PATTERNS
        x[r] = 0
        if p == 4:                                    # all logits equal (= bias): x row zero
            continue
        x[r, p] = 1.0
        if p == 0:                                    # all top-8 in one tile: 10 large values in groups of ties
            base = (ft // 2) * TILE + min(40, max(0, F - (ft // 2) * TILE - 10))
            n = min(10, F - base)
            W[p, base:base + n] = torch.tensor([(64 + j2 % 5) / 16 for j2 in range(n)])
        elif p == 1:                                  # one winner per tile
            for t in range(ft):
                W[p, min(F - 1, t * TILE + (37 * t) % TILE)] = 4.0
        elif p == 2:                                  # the row maximum at the last valid feature of the last tile
            W[p, F - 1] = 6.0
        elif p == 3:                                  # equal logits across the tile boundary 127 / 128 and inside a tile
            pairs = [(127, 128), (300, 310)] if F > 310 else [(2, 5)]
            for a, b in pairs:
                W[p, a] = W[p, b] = 5.0
                if bias is not None:
                    bias[b] = bias[a]


def proj_inputs(R, K, F, exact, has_bias, first, seed):
    g = gen(seed)
    if exact:
        x = torch.randint(-8, 9, (R, K), generator=g).float() / 8
        W = torch.randint(-2, 3, (K, F), generator=g).float() / 16
        bias = torch.randint(-16, 17, (F,), generator=g).float() / 128 if has_bias else None
    else:
        x = torch.randn(R, K, generator=g)
        W = torch.randn(K, F, generator=g) / np.sqrt(K) * 3
        bias = torch.randn(F, generator=g) * 0.5 if has_bias else None
    rows = sorted({R - 1, 0, R // 2, min(R - 1, 129), min(R - 1, 255)}, key=lambda r: (r != R - 1, r))
    plant(x, W, bias, F, rows[:N_PATTERNS], first)
    return x, W, bias


@pytest.mark.parametrize("case", PROJ_CASES, ids=[c[0] for c in PROJ_CASES])
def test_vocab_stats_against_fp64(case):
    from fpnmt.engine import vocab_stats
    name, R, K, F, exact, has_bias, first = case
    x, W, bias = proj_inputs(R, K, F, exact, has_bias, first, seed=zlib.crc32(name.encode()))
    ft = (F + TILE - 1) // TILE
    extra = 5                                          # poisoned rows >= R
    stat = torch.full((R + extra, ft, 2), float("nan"), device="cuda")
    val = torch.full((R + extra, ft, 8), float("nan"), device="cuda")
    idx = torch.full((R + extra, ft, 8), SENTINEL_ID, dtype=torch.int32, device="cuda")
    vocab_stats(x.cuda(), W.numpy(), None if bias is None else bias.numpy(), stat=stat, val=val, idx=idx)
    stat, val, idx = stat.cpu(), val.cpu(), idx.cpu()
    assert bool(torch.isnan(stat[R:]).all()) and bool(torch.isnan(val[R:]).all()) and bool((idx[R:] == SENTINEL_ID).all()), \
        "%s: rows >= R were written" % name
    stat, val, idx = stat[:R].double().numpy(), val[:R].double().numpy(), idx[:R].numpy().astype(np.int64)

    xq = q_act(x, "bf16").double()
    Wq = W.to(torch.bfloat16).double()
    b = torch.zeros(F, dtype=torch.float64) if bias is None else bias.double()
    z = (xq @ Wq + b).numpy()
    m, S, vref, iref, t, D = tile_reference(z, F)
    bS = sumexp_bound(S, t, D)
    if exact:
        assert np.abs(z).max() * 128 < 2 ** 17
        assert np.array_equal(stat[..., 0], m), "%s: tile maxima differ at %s" % (name, np.argwhere(stat[..., 0] != m)[:5])
        assert np.array_equal(val, vref), "%s: candidate values differ at %s" % (name, np.argwhere(val != vref)[:5])
        bad = np.argwhere(idx != iref)
        assert bad.size == 0, "%s: candidate ids differ at (row, tile, rank) %s: %s vs %s" % (
            name, bad[:5].tolist(), idx[tuple(bad[0])] if bad.size else None, iref[tuple(bad[0])] if bad.size else None)
        err = np.abs(stat[..., 1] - S)
        record("vocab_stats.sumexp (exact inputs)", float((err / bS).max()), 1.0)
        assert (err <= bS).all(), "%s: sum exp off by %.3g > bound %.3g" % (name, err.max(), bS[np.unravel_index((err / bS).argmax(), err.shape)])
        return
    # random inputs: fp32 accumulation bound delta per logit, taken per tile as its maximum
    absacc = (xq.abs() @ Wq.abs()).numpy()
    delta = K * 2.0 ** -23 * absacc + U * np.abs(z)
    dp = np.zeros((R, ft * TILE))
    dp[:, :F] = delta
    dt = dp.reshape(R, ft, TILE).max(-1)
    for what, got, ref, bnd in (("max", stat[..., 0], m, dt), ("values", val, vref, dt[..., None])):
        err = np.abs(got - ref)
        record("vocab_stats.%s (random inputs)" % what, float((err / bnd).max()), 1.0)
        assert (err <= bnd).all(), "%s: %s off by %.3g" % (name, what, float((err - bnd).max()))
    bSr = bS + S * np.expm1(2 * dt)
    err = np.abs(stat[..., 1] - S)
    record("vocab_stats.sumexp (random inputs)", float((err / bSr).max()), 1.0)
    assert (err <= bSr).all(), "%s: sum exp off" % name
    gap_prev = np.concatenate([np.full((R, ft, 1), np.inf), vref[..., :-1] - vref[..., 1:]], -1)
    gap_next = np.concatenate([vref[..., :-1] - vref[..., 1:], np.full((R, ft, 1), np.inf)], -1)
    # the 9th value of the tile bounds the gap of rank 8 from below
    zt = np.full((R, ft * TILE), -np.inf)
    zt[:, :F] = z
    ninth = -np.sort(-zt.reshape(R, ft, TILE), -1)[..., NC]
    gap_next[..., -1] = vref[..., -1] - ninth
    clear = (gap_prev > 2 * dt[..., None]) & (gap_next > 2 * dt[..., None])
    assert clear.mean() > 0.5, "%s: too few separated candidates (%.2f)" % (name, clear.mean())
    assert np.array_equal(idx[clear], iref[clear]), "%s: candidate ids differ" % name


# ------------------------------------------------------------------------------------------------------------------------
# (b) the beam step's merge of the partials
_WEIGHTS = {}


def make_engine(B, N, V, **kw):
    from fpnmt.engine import Engine
    from fpnmt.weights import init_weights
    if V not in _WEIGHTS:
        _WEIGHTS[V] = init_weights("mobilenet224_1.0", vocab=V, seed=0, num_layers=1)
    return Engine(_WEIGHTS[V], backbone="mobilenet224_1.0", batch=B, beam=N, vocab=V, max_len=4, num_layers=1, image_size=256,
                  use_graphs=False, **kw)


# N, B, V (+ engine options)
MERGE_CASES = [
    (1, 3, 256, {}),
    (2, 1, 24576, {}),
    (2, 3, 1000, {}),
    (4, 3, 10000, {}),
    (4, 1, 8, {}),
    (8, 3, 256, {}),
    (8, 1, 1000, {}),
    (8, 3, 24576, {}),
    (8, 3, 8, {}),
    (8, 3, 1000, {"finished_beams": True, "length_penalty": 0.6}),
]
TRIALS = ["random", "identical_rows", "ties_across_tiles", "top_n_in_one_tile", "spread_winners", "peaked", "dead_beams",
          "fewer_tokens_than_beams"]


def merge_inputs(trial, B, N, V, seed):
    """(logits (rows, V) fp32, scores (rows,), number of valid tokens)."""
    g = gen(seed)
    rows = B * N
    logits = torch.randn(rows, V, generator=g) * (3.0 if trial == "peaked" else 1.0)
    scores = -torch.rand(rows, generator=g) * 3
    vv = V
    if trial == "identical_rows":                     # the reference's start state (pipeline.py:101-102)
        logits = logits.reshape(B, N, V)[:, :1].repeat(1, N, 1).reshape(rows, V)
        scores = torch.zeros(rows)
    elif trial == "ties_across_tiles":
        a, b = (127, 128) if V > 128 else (2, 5)
        logits[:, a] = logits[:, b] = logits.max() + 1
    elif trial == "top_n_in_one_tile":
        t0 = ((V + TILE - 1) // TILE) // 2
        for j in range(N):
            logits[:, min(V - 1, t0 * TILE + 3 + j)] = logits.max() + 1 + 0.01 * j
    elif trial == "spread_winners":                   # each of the N best tokens alone in its tile
        nt = (V + TILE - 1) // TILE
        for j in range(min(N, nt)):
            logits[:, min(V - 1, j * TILE + 17)] = 6.0 - 0.25 * j
    elif trial == "dead_beams":                       # the true-beam start state: beams 1..N-1 dead
        scores.reshape(B, N)[:, 1:] = -float("inf")
    elif trial == "fewer_tokens_than_beams":
        vv = max(1, N // 2)
        logits[:, vv:] = -float("inf")
        scores -= 100.0                               # below whatever an earlier call left in the candidate buffers
    return logits, scores, vv


@pytest.mark.parametrize("N,B,V,kw", MERGE_CASES, ids=["N%d_B%d_V%d%s" % (n, b, v, "_finished" if k else "") for n, b, v, k in MERGE_CASES])
def test_beam_step_vstats_against_oracle(N, B, V, kw):
    eng = make_engine(B, N, V, **kw)
    try:
        for i, trial in enumerate(TRIALS):
            if trial == "fewer_tokens_than_beams" and N < 2:
                continue
            logits, scores, vv = merge_inputs(trial, B, N, V, seed=1000 * N + 10 * B + i + V)
            stat, val, idx = host_partials(logits, vv)
            par, tok, sc = [t.cpu().numpy() for t in eng.beam_step_vstats(stat.cuda(), val.cuda(), idx.cuda(), scores.cuda())]
            lpar, ltok, lsc = [t.cpu().numpy() for t in eng.beam_step(logits.cuda(), scores.cuda())]
            assert np.array_equal(par, lpar) and np.array_equal(tok, ltok), (trial, par, lpar, tok, ltok)
            z = logits[:, :vv].double().numpy()
            s64 = scores.double().numpy()
            m_t, S_t = stat[..., 0].double().numpy(), stat[..., 1].double().numpy()
            lse, eps, logsum = lse_terms(m_t, S_t, U)
            lse_l = z.max(-1) + np.log(np.exp(z - z.max(-1, keepdims=True)).sum(-1))
            eps_l = logits_path_eps(z)
            for b in range(B):
                sl = slice(b * N, (b + 1) * N)
                p, t, _ = O.beam_step(logits[sl, :vv].numpy(), scores[sl].numpy(), "log")
                assert np.array_equal(par[sl], p) and np.array_equal(tok[sl], t), (trial, b, par[sl], p, tok[sl], t)
                r = b * N + p                               # the chosen parents' rows
                zz = z[r, t]
                exact = s64[r] + zz - lse_l[r]
                bv = merge_bound(lse[r], eps[r], logsum[r], zz, s64[r])
                bl = merge_bound(lse_l[r], eps_l[r], logsum[r], zz, s64[r])
                fin = np.isfinite(exact)
                assert np.array_equal(np.isfinite(sc[sl]), fin) and np.array_equal(np.isfinite(lsc[sl]), fin), trial
                for what, got, bnd in (("beam_step_vstats.score", sc[sl], bv), ("beam_step.score (logits path)", lsc[sl], bl)):
                    err = np.abs(got[fin] - exact[fin])
                    if err.size:
                        record(what, float((err / bnd[fin]).max()), 1.0)
                        assert (err <= bnd[fin]).all(), "%s %s image %d: %s off by %s > %s" % (trial, what, b, got, err, bnd[fin])
                err = np.abs(sc[sl][fin] - lsc[sl][fin])
                if err.size:
                    record("beam_step_vstats vs logits path", float((err / (bv + bl)[fin]).max()), 1.0)
                    assert (err <= (bv + bl)[fin]).all(), (trial, b, sc[sl], lsc[sl])
    finally:
        eng.close()


# ------------------------------------------------------------------------------------------------------------------------
# (c) projection -> merge
@pytest.mark.parametrize("N,B,V", [(8, 3, 1000), (4, 3, 10000)])
@pytest.mark.parametrize("identical", [False, True])
def test_projection_then_merge_equals_oracle(N, B, V, identical):
    from fpnmt.engine import vocab_stats
    rows, K = B * N, 512
    x, W, bias = proj_inputs(rows, K, V, True, True, 0, seed=V + N + identical)
    g = gen(V + N)
    scores = -torch.rand(rows, generator=g) * 3
    if identical:
        x = x.reshape(B, N, K)[:, :1].repeat(1, N, 1).reshape(rows, K)
        scores = torch.zeros(rows)
    z = (x.double() @ W.double() + bias.double()).numpy()
    logits = torch.from_numpy(z.astype(np.float32))
    assert np.array_equal(logits.double().numpy(), z)
    stat, val, idx = vocab_stats(x.cuda(), W.numpy(), bias.numpy())
    eng = make_engine(B, N, V)
    try:
        par, tok, sc = [t.cpu().numpy() for t in eng.beam_step_vstats(stat, val, idx, scores.cuda())]
    finally:
        eng.close()
    m, S, _, _, t, D = tile_reference(z, V)
    e_t = sumexp_bound(S, t, D) / S
    lse, eps, logsum = lse_terms(m, S, e_t)
    s64 = scores.double().numpy()
    for b in range(B):
        sl = slice(b * N, (b + 1) * N)
        p, tt, _ = O.beam_step(logits[sl].numpy(), scores[sl].numpy(), "log")
        assert np.array_equal(par[sl], p) and np.array_equal(tok[sl], tt), (b, par[sl], p, tok[sl], tt)
        r = b * N + p
        exact = s64[r] + z[r, tt] - lse[r]
        bnd = merge_bound(lse[r], eps[r], logsum[r], z[r, tt], s64[r])
        err = np.abs(sc[sl] - exact)
        record("projection -> merge score", float((err / bnd).max()), 1.0)
        assert (err <= bnd).all(), (b, sc[sl], exact, bnd)


# ------------------------------------------------------------------------------------------------------------------------
# (d) contract: refusals return an error code and a message, and launch nothing
def test_refusals_launch_nothing():
    from fpnmt import _lib
    from fpnmt.engine import vocab_stats

    def refused(fn, needle):
        with pytest.raises(_lib.FpnmtError) as e:
            fn()
        assert e.value.code == _lib.ERR_INVALID and needle in str(e.value), str(e.value)

    def partials(rows, tiles):
        return (torch.zeros(rows, tiles, 2, device="cuda"), torch.full((rows, tiles, 8), -float("inf"), device="cuda"),
                torch.full((rows, tiles, 8), PAD_ID, dtype=torch.int32, device="cuda"))

    for N, kw in ((4, {"score_mode": "prob"}), (9, {}), (4, {})):
        eng = make_engine(1, N, 1000, **kw)
        try:
            n0 = eng.launch_count
            sc = torch.zeros(N, device="cuda")
            if N == 4 and not kw:
                refused(lambda: eng.beam_step_vstats(*partials(N, 193), sc), "192 vocabulary tiles")
                st, vl, ix = partials(N, 8)
                out = [torch.empty(N, dtype=dt, device="cuda") for dt in (torch.int32, torch.int32, torch.float32)]
                refused(lambda: _lib.check(eng.lib.fpnmt_beam_step_vstats(eng._h, st.data_ptr(), vl.data_ptr(), ix.data_ptr(), 0,
                                                                          sc.data_ptr(), *[o.data_ptr() for o in out],
                                                                          torch.cuda.current_stream().cuda_stream)),
                        "192 vocabulary tiles")
            else:
                refused(lambda: eng.beam_step_vstats(*partials(N, 8), sc), "log scores, beam <= 8")
            torch.cuda.synchronize()
            assert eng.launch_count == n0
        finally:
            eng.close()
    x = torch.zeros(4, 512, device="cuda")
    refused(lambda: vocab_stats(x, np.zeros((512, 1000), np.float32), precision="bf16x3"), "bf16-mode kernel")
    refused(lambda: vocab_stats(x, np.zeros((512, 1004), np.float32)), "multiples of 8")
