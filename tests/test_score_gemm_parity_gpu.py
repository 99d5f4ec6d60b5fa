"""The score GEMM (csrc/scoring.cu) against a float64 reference of the same float32 inputs, entry by entry.

``score_matrix(E, T, r, q, cst, alpha)`` is ``alpha * (r_i + q_j + cst) + alpha * E_i . T_j``; the reference computes
exactly that in float64 on the device.  Every entry is checked against its own bound, built from ``A = |E| |T|^T`` (float64),
the row norms, the l1 row norms and the operand maxima, and every bound is checked to be tight enough: the same
comparison made against a deliberately wrong reference (or with the single-pass result against the three-pass bound)
must fail (``_controls``).

How the GEMM computes (csrc/scoring.cu, operand preparation): each operand X is scaled by a power of two 2^s so that its
largest entry lies in [2^9, 2^10), and rounded to fp16, ``hi = fl16(X 2^s)``.  Products of two fp16 values are exact in
fp32; the tensor core accumulates them in fp32 in K steps of 16.  The three-pass mode also keeps ``lo = fl16(X 2^s - hi)``
and accumulates hi*hi + hi*lo + lo*hi.  Per entry x of an operand with maximum M (unscaled units):

* fp16 rounding of a normal value: ``|hi - x| <= 2^-11 |x|``.  fp16 subnormals are spaced 2^-24, so a scaled value
  below 2^-14 is off by up to 2^-25, which is ``2^-25 2^-s <= 2^-34 M`` unscaled (2^s >= 2^9 / M).  Hence
  ``|hi - x| <= 2^-11 |x| + 2^-34 M``.
* One pass: ``|e t - hi_e hi_t| <= (2^-10 + 2^-22) |e| |t| + 2^-34 (1 + 2^-10) (M_T |e| + M_E |t|)`` (dropping a
  2^-68 M_E M_T term).  Summed over k: ``(2^-10 + 2^-22) A_ij + SUB_ij`` with
  ``SUB_ij = 2^-34 (1 + 2^-10) (M_T |E_i|_1 + M_E |T_j|_1)``.
* Three passes: ``x = hi + lo + d`` with ``|d| <= 2^-22 |x| + 2^-34 M`` (``x 2^s - hi`` is exact in fp32, its fp16
  rounding is the error) and ``|lo| <= 2^-11 (1 + 2^-11) |x| + 2^-34 M``.  The computed product misses ``lo_e lo_t`` and
  carries ``e d_t + t d_e``, so ``|e t - c| <= 3 (1 + 2^-10) 2^-22 |e| |t| + SUB terms``: ``PROD3 = 3.003 2^-22 A_ij + SUB_ij``.
* fp32 accumulation: ``n = passes * Dp / 16`` accumulator updates.  Two parts, constants measured on the B200: a part
  that grows linearly with n, at most ``C_LIN`` units of 2^-24 of the entry's magnitude per update (partial sums that
  grow monotonically, e.g. all-negative rows), and a random-walk part, ``C_RW 2^-24 sqrt(n) |E_i|_2 |T_j|_2``, for
  partial sums of either sign (Cauchy-Schwarz bounds every partial sum by ``|E_i|_2 |T_j|_2``).
* The epilogue: alpha and ``alpha * cst`` are rounded to float32, then one product, one FMA and one sum (csrc/scoring.cu,
  fast and generic paths alike): at most ``C_EPI`` units of 2^-24 of ``|alpha| (|E_i . T_j| + |r_i| + |q_j| + |cst|) +
  |S_ij|``.

``bound = |alpha| (PROD + ACC) + EPI``.  A float16 output is checked against the same bound plus half an fp16 ulp of the entry.
"""
import math

import numpy
import pytest
import torch

import sidekit_b200 as sk
from sidekit_b200 import synth
from sidekit_b200.iv_scoring import PackedEmbeddings, TrialIndex, score_trials, _simplified_plda_terms

C_LIN = 1.0
C_RW = 4.0
C_EPI = 6.0

SWEEP_D = (1, 3, 8, 17, 63, 64, 65, 100, 128, 129, 191, 192, 200, 255, 256, 257, 300, 384, 512, 520, 1024, 2048)
SHAPES = ((1, 1), (1, 129), (127, 128), (128, 257), (129, 31), (333, 517), (1100, 700))
PASSES = (1, 3)
TOPK_D = (100, 150, 192, 300)
TOPK_K = (5, 32, 100)                    # k <= 32: the GEMM's top-k epilogue; k > 32: score panels + select


def variant(D, passes, mode):
    """The kernel body ``gemm_packed`` (csrc/scoring.cu) runs for width D, a forced pass count and an output mode
    ("matrix", "trials" or "topk" for the fused top-k epilogue, k <= 32): ``(mode, layout, passes)`` with layout "KC128" /
    "KC64" (the E panel resident in tensor memory, 128- or 64-wide K stages) or "stream" (both operands streamed).  None
    where the call is rejected."""
    Dp = -(-D // 64) * 64
    if Dp > 256:
        if mode == "trials":
            return None
        return ("matrix", "stream", passes)            # top-k of a wide operand takes the score-panel path
    return (mode, "KC128" if Dp % 128 == 0 else "KC64", passes)


ALL_BODIES = {(m, l, p) for p in PASSES for m, l in (("matrix", "KC128"), ("matrix", "KC64"), ("matrix", "stream"),
                                                      ("trials", "KC128"), ("trials", "KC64"), ("topk", "KC128"),
                                                      ("topk", "KC64"))}


def test_the_parametrisation_reaches_every_kernel_body():
    reached = {variant(D, p, "matrix") for D in SWEEP_D for p in PASSES}
    reached |= {variant(D, p, "trials") for D in SWEEP_D for p in PASSES} - {None}
    reached |= {variant(D, p, "topk" if k <= 32 else "matrix") for D in TOPK_D for k in TOPK_K for p in PASSES}
    assert len(ALL_BODIES) == 14
    assert reached == ALL_BODIES, sorted(ALL_BODIES - reached)


# ----------------------------------------------------------------------------------------------------------- operands
def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def operand(kind, n, D, seed):
    """(n, D) float32 CUDA operand: "unit" / "gauss" rows, "scaled" (N(0,1) rows times 1e-3 .. 1e3: small rows reach fp16
    subnormals after the operand's scaling), "zero", "negative" (-|N(0,1)|), "plda" ((e - mu) Psi of unit rows, synth_plda),
    "repeated" (every entry of a row +-1/sqrt(D): coherent fp16 rounding errors)."""
    x = torch.randn((n, D), generator=_gen(seed), device="cuda", dtype=torch.float64)
    if kind == "unit":
        x = x / x.norm(dim=1, keepdim=True)
    elif kind == "scaled":
        x = x * torch.logspace(-3, 3, n, device="cuda", dtype=torch.float64)[torch.randperm(n, generator=_gen(seed + 7), device="cuda")][:, None]
    elif kind == "zero":
        x = torch.zeros_like(x)
    elif kind == "negative":
        x = -x.abs()
    elif kind == "plda":
        mu, F, Sigma = synth.synth_plda(D, D, seed=seed % 1000)
        _, Psi, _ = _simplified_plda_terms(F, Sigma, 1.0)
        x = x / x.norm(dim=1, keepdim=True)
        x = (x - torch.from_numpy(mu).cuda()) @ torch.from_numpy(Psi).cuda()
    elif kind == "repeated":
        x = torch.sign(x[:, :1]).expand(n, D) / math.sqrt(D)
    elif kind != "gauss":
        raise ValueError(kind)
    return x.float().contiguous()


def _vec(n, seed, present=True, misaligned=False):
    """Per-row term: None, an N(0,1) float32 vector, or one at a 4-byte-misaligned base."""
    if not present:
        return None
    v = torch.randn((n + 1,), generator=_gen(seed), device="cuda").float()
    return v[1:] if misaligned else v[:n].contiguous()


# ---------------------------------------------------------------------------------------------- reference and bound
def reference(E, T, r, q, cst, alpha, passes, k_cols=None):
    """(ref, bound) float64 (Ne, Nt): the float64 score and the per-entry error bound of the module docstring for a
    forced pass count (passes = 0 is checked against the single-pass bound, which also covers three passes).  ``k_cols``: use only
    the first k_cols columns of E and T for the reference (a control; the bound stays that of the full operands)."""
    D = E.shape[1]
    E64, T64 = E.double(), T.double()
    k = D if k_cols is None else k_cols
    dot = E64[:, :k] @ T64[:, :k].T
    terms = torch.full_like(dot, float(cst))
    terms_abs = torch.full_like(dot, abs(float(cst)))
    if r is not None:
        terms += r.double()[:, None]
        terms_abs += r.double().abs()[:, None]
    if q is not None:
        terms += q.double()[None, :]
        terms_abs += q.double().abs()[None, :]
    ref = alpha * terms + alpha * dot
    dot_full = dot if k == D else E64 @ T64.T
    A = E64.abs() @ T64.abs().T
    mE, mT = E64.abs().max(), T64.abs().max()
    sub = 2.0 ** -34 * (1 + 2.0 ** -10) * (mT * E64.abs().sum(1)[:, None] + mE * T64.abs().sum(1)[None, :])
    if passes == 3:
        prod, combos = 3.003 * 2.0 ** -22 * A + sub, 3
    else:
        prod, combos = (2.0 ** -10 + 2.0 ** -22) * A + sub, 1
    n_acc = combos * (-(-D // 64) * 64) // 16
    acc = 2.0 ** -24 * (C_LIN * n_acc * dot_full.abs() + C_RW * math.sqrt(n_acc) * E64.norm(dim=1)[:, None] * T64.norm(dim=1)[None, :])
    epi = C_EPI * 2.0 ** -24 * (abs(alpha) * (dot_full.abs() + terms_abs) + ref.abs())
    return ref, abs(alpha) * (prod + acc) + epi


def _half_ulp16(x):
    """Half an fp16 ulp of |x| (float64), 2^-25 in the subnormal range."""
    e = torch.floor(torch.log2(x.abs().clamp_min(2.0 ** -14)))
    return torch.exp2(e - 11)


def excess(out, ref, bound):
    """max over entries of |out - ref| / bound (float64); > 1 means some entry is out of its bound."""
    err = (out.double() - ref).abs()
    if out.dtype == torch.float16:
        bound = bound + _half_ulp16(ref.abs() + bound)
    return (err / bound.clamp_min(1e-300)).max().item() if err.numel() else 0.0


# ------------------------------------------------------------------------------------------------- output layouts
_SENTINEL = {torch.float32: (torch.int32, 0x7fc0beef), torch.float64: (torch.int64, 0x7ff8dead0000beef),
             torch.float16: (torch.int16, 0x7e5a)}


def output_view(Ne, Nt, dtype, layout):
    """(out, flat, inside): an (Ne, Nt) view into a NaN-sentinel-filled buffer ``flat``, with row stride Nt ("plain"),
    Nt + 5 ("ld5"), Nt + 8 ("ld8"), or Nt at a base 4 bytes past an aligned address ("misaligned"; 8 bytes for float64);
    ``inside`` marks the elements of ``flat`` the view covers."""
    ld = {"plain": Nt, "ld5": Nt + 5, "ld8": Nt + 8, "misaligned": Nt}[layout]
    off = 0 if layout != "misaligned" else (2 if dtype == torch.float16 else 1)
    n = off + Ne * ld + 3
    itype, bits = _SENTINEL[dtype]
    flat = torch.full((n,), bits, dtype=itype, device="cuda").view(dtype)
    out = flat[off:off + Ne * ld].view(Ne, ld)[:, :Nt]
    inside = torch.zeros((n,), dtype=torch.bool, device="cuda")
    inside[off:off + Ne * ld].view(Ne, ld)[:, :Nt] = True
    return out, flat, inside


def sentinel_kept(flat, inside):
    itype, bits = _SENTINEL[flat.dtype]
    return bool((flat.view(itype)[~inside] == bits).all())


# ---------------------------------------------------------------------------------------------------- matrix sweep
# (E kind, T kind, alpha, cst, row term, column term ("none" / "plain" / "misaligned"), passes, out dtype, out layout)
CASES = (
    ("unit", "unit", 1.0, 0.0, False, "none", 3, torch.float32, "plain"),
    ("unit", "unit", 1.0, 0.0, False, "none", 1, torch.float32, "ld5"),
    ("gauss", "gauss", -2.0, 0.5, True, "plain", 0, torch.float32, "ld8"),
    ("scaled", "unit", 0.37, -1.25, True, "misaligned", 3, torch.float64, "plain"),
    ("unit", "scaled", 1.0, 0.0, False, "plain", 0, torch.float64, "misaligned"),
    ("zero", "gauss", -2.0, 0.75, True, "plain", 3, torch.float32, "misaligned"),
    ("negative", "negative", 0.37, 0.0, False, "none", 1, torch.float32, "ld5"),
    ("plda", "unit", 1.0, -3.0, True, "plain", 0, torch.float32, "plain"),
    ("unit", "unit", -2.0, 0.25, True, "misaligned", 1, torch.float16, "ld8"),
    ("unit", "unit", 0.37, 0.0, False, "none", 3, torch.float16, "misaligned"),
)


def matrix_case(D, shape, case, seed):
    """Runs one ``score_matrix`` case; returns (out, ref, bound, sentinel intact)."""
    ek, tk, alpha, cst, row, col, passes, dtype, layout = case
    Ne, Nt = shape
    E, T = operand(ek, Ne, D, seed), operand(tk, Nt, D, seed + 1)
    r = _vec(Ne, seed + 2, row)
    q = _vec(Nt, seed + 3, col != "none", col == "misaligned")
    out, flat, inside = output_view(Ne, Nt, dtype, layout)
    got = sk.score_matrix(E, T, r, q, cst=cst, alpha=alpha, passes=passes, out_dtype=dtype, out=out)
    assert got.data_ptr() == out.data_ptr()
    ref, bound = reference(E, T, r, q, cst, alpha, passes)
    return out, ref, bound, sentinel_kept(flat, inside)


def _case_plan(D):
    """The (shape, case) pairs run at width D: every case once, the shapes rotated with D; the PLDA fold (a host D x D
    inverse) up to D = 520."""
    di = SWEEP_D.index(D)
    plan = []
    for c, case in enumerate(CASES):
        if case[0] == "plda" and D > 520:
            continue
        plan.append((SHAPES[(di + c) % len(SHAPES)], case))
    return plan


@pytest.mark.gpu
@pytest.mark.parametrize("D", SWEEP_D)
def test_score_matrix_within_the_bound_of_every_entry(D):
    for i, (shape, case) in enumerate(_case_plan(D)):
        out, ref, bound, kept = matrix_case(D, shape, case, seed=1000 * D + i)
        ex = excess(out, ref, bound)
        assert ex <= 1.0, (D, shape, case, ex)
        assert kept, ("entries outside the output view were written", D, shape, case)


def _controls(D, seed=7):
    """The bound's negative controls on unit rows (333 x 517, row and column terms): each entry of the returned dict is
    the excess (``excess``) of a comparison that must FAIL (> 1), plus "ok1" / "ok3", the excess of the real comparisons,
    which must pass."""
    Ne, Nt, alpha, cst = 333, 517, 1.0, 0.5
    E, T = operand("unit", Ne, D, seed), operand("unit", Nt, D, seed + 1)
    r, q = _vec(Ne, seed + 2), _vec(Nt, seed + 3)
    out = {p: sk.score_matrix(E, T, r, q, cst=cst, alpha=alpha, passes=p) for p in PASSES}
    res = {}
    for p in PASSES:
        ref, bound = reference(E, T, r, q, cst, alpha, p)
        res["ok%d" % p] = excess(out[p], ref, bound)
        tail, _ = reference(E, T, r, q, cst, alpha, p, k_cols=max(0, D - 8))
        res["k_tail%d" % p] = excess(out[p], tail, bound)
        shifted, _ = reference(E, T, r, torch.roll(q, 1), cst, alpha, p)
        res["col_shift%d" % p] = excess(out[p], shifted, bound)
        if p == 3 and not torch.equal(out[1], out[3]):
            res["one_pass_vs_bound3"] = excess(out[1], ref, bound)
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("D", SWEEP_D)
def test_bounds_are_tight_enough_to_catch_a_lost_k_tail_a_shifted_column_term_and_a_dropped_split_product(D):
    res = _controls(D)
    assert res["ok1"] <= 1.0 and res["ok3"] <= 1.0, res
    for name, ex in res.items():
        if not name.startswith("ok"):
            assert ex > 1.0, (D, name, res)
    if D > 1:      # unit rows of one column are +-1, exact in fp16: both pass counts give the same bits
        assert "one_pass_vs_bound3" in res


@pytest.mark.gpu
@pytest.mark.parametrize("D,shape", [(192, (2000, 3000)), (300, (2000, 3000))])
def test_grids_of_more_tiles_than_ctas(D, shape):
    """384 (row panel, column tile) items over 148 CTAs: runs that cross row-panel boundaries."""
    for p in PASSES:
        out, ref, bound, kept = matrix_case(D, shape, ("unit", "gauss", -2.0, 0.5, True, "plain", p, torch.float32, "ld5"), seed=5 + p)
        assert excess(out, ref, bound) <= 1.0 and kept, p


@pytest.mark.gpu
@pytest.mark.parametrize("D", SWEEP_D)
def test_packed_test_side_is_bit_identical_to_the_plain_call(D):
    Ne, Nt = SHAPES[SWEEP_D.index(D) % len(SHAPES)]
    E, T = operand("gauss", Ne, D, 31), operand("unit", Nt, D, 32)
    r, q = _vec(Ne, 33), _vec(Nt, 34, misaligned=True)
    P = PackedEmbeddings(T)
    for p in (0, 1, 3):
        for dtype in (torch.float32, torch.float16):
            want = sk.score_matrix(E, T, r, q, cst=0.25, alpha=-2.0, passes=p, out_dtype=dtype)
            got = sk.score_matrix(E, P, r, q, cst=0.25, alpha=-2.0, passes=p, out_dtype=dtype)
            assert torch.equal(got, want), (p, dtype)


# ----------------------------------------------------------------------------------------------------- trial lists
@pytest.mark.gpu
@pytest.mark.parametrize("D", SWEEP_D)
def test_trial_list_mode_against_the_float64_reference(D):
    Ne, Nt = (333, 517) if D % 2 else (129, 31)
    E, T = operand("unit", Ne, D, 41), operand("gauss", Nt, D, 42)
    r, q = _vec(Ne, 43), _vec(Nt, 44, misaligned=D % 3 == 0)
    mask = torch.rand((Ne, Nt), generator=_gen(45), device="cuda") < 0.3
    if variant(D, 1, "trials") is None:
        with pytest.raises(RuntimeError, match="trial-list mode supports embeddings of up to 256 dimensions"):
            score_trials(E, T, mask, r, q, cst=0.5, alpha=0.37, passes=3)
        return
    idx = TrialIndex(mask)
    for p in PASSES:
        got = score_trials(E, T, idx, r, q, cst=0.5, alpha=0.37, passes=p)
        ref, bound = reference(E, T, r, q, 0.5, 0.37, p)
        assert got.shape == (int(mask.sum()),)
        assert excess(got, ref[mask], bound[mask]) <= 1.0, p
        assert torch.equal(score_trials(E, PackedEmbeddings(T), idx, r, q, cst=0.5, alpha=0.37, passes=p), got)


# ------------------------------------------------------------------------------------------------------------- top-k
@pytest.mark.gpu
@pytest.mark.parametrize("k", TOPK_K)
@pytest.mark.parametrize("D", TOPK_D)
def test_topk_values_are_score_matrix_entries_and_indices_follow_the_float64_order(D, k):
    Ne, Nt = 333, 517
    E, T = operand("unit", Ne, D, 51), operand("unit", Nt, D, 52)
    r, q = _vec(Ne, 53), 0.05 * _vec(Nt, 54)
    checked = 0
    for p in PASSES:
        S = sk.score_matrix(E, T, r, q, cst=0.5, alpha=-2.0, passes=p)
        vals, idx = sk.score_topk(E, T, k, r, q, cst=0.5, alpha=-2.0, passes=p)
        assert torch.equal(vals, torch.gather(S, 1, idx))
        assert torch.equal(vals, torch.sort(S, dim=1, descending=True).values[:, :k])
        ref, bound = reference(E, T, r, q, 0.5, -2.0, p)
        rs, ri = torch.sort(ref, dim=1, descending=True)
        gap = 2.0 * bound.max(dim=1, keepdim=True).values
        above = torch.cat([torch.full_like(rs[:, :1], math.inf), rs[:, :-1] - rs[:, 1:]], dim=1)[:, :k]
        below = (rs[:, :-1] - rs[:, 1:])[:, :k] if Nt > k else torch.full_like(rs[:, :k], math.inf)
        clear = (above > gap) & (below > gap)
        assert torch.equal(idx[clear], ri[:, :k][clear]), p
        checked += int(clear.sum())
    assert checked > Ne        # the comparison is not vacuous


# --------------------------------------------------------------------------------------------------------- as-norm
@pytest.mark.gpu
@pytest.mark.parametrize("C,top_k", [(C, k) for C in (2, 200, 5994, 51200) for k in sorted({2, 200, C}) if k <= C])
def test_asnorm_statistics_are_exact_over_the_float32_scores(C, top_k):
    """Mean and unbiased std of the top_k cohort scores of every row, against torch.topk in float64 over the same float32
    scores; the cohort repeats its rows (exactly tied scores across the threshold) and scores of both signs occur."""
    from sidekit_b200 import bulk
    N, D = 257, 192
    X = operand("unit", N, D, 61)
    base = operand("unit", max(1, C // 3), D, 62)
    coh = base[torch.randint(0, base.shape[0], (C,), generator=_gen(63), device="cuda")].contiguous()
    mean, std = bulk._asnorm_stats_cuda(X, coh, top_k)
    S = sk.score_matrix(X, coh, passes=3).double()
    assert (S < 0).any()
    top = torch.topk(S, top_k, dim=1).values
    assert torch.equal(mean, top.mean(dim=1).float())
    assert torch.allclose(std.double(), top.std(dim=1), rtol=2.0 ** -22, atol=1e-30)


@pytest.mark.gpu
def test_asnorm_statistics_reject_a_cohort_beyond_the_shared_memory_limit():
    from sidekit_b200 import bulk
    X, coh = operand("unit", 4, 64, 1), operand("unit", 51201, 64, 2)
    with pytest.raises(RuntimeError, match="C <= 51200"):
        bulk._asnorm_stats_cuda(X, coh, 200)


@pytest.mark.gpu
@pytest.mark.parametrize("D", (100, 300))
def test_asnorm_apply_against_the_float64_formula(D):
    """The as-norm epilogue (a column term that multiplies the accumulator): 0.5 (s - m_i) / s_i + 0.5 (s - m_j) / s_j."""
    from sidekit_b200 import _lib, bulk
    N = 1000
    X = operand("unit", N, D, 71)
    g = _gen(72)
    mean = (0.2 * torch.rand((N,), generator=g, device="cuda") - 0.1).float()
    std = (0.05 + 0.15 * torch.rand((N,), generator=g, device="cuda")).float()
    ref, bound = reference(X, X, None, None, 0.0, 1.0, 3)
    dot, dot_bound = ref, bound
    m, s = mean.double(), std.double()
    mul = 0.5 / s[:, None] + 0.5 / s[None, :]
    want = dot * mul - 0.5 * m[:, None] / s[:, None] - 0.5 * m[None, :] / s[None, :]
    bound = mul * dot_bound + C_EPI * 2.0 ** -24 * (mul * dot.abs() + 0.5 * (m / s).abs()[:, None] + 0.5 * (m / s).abs()[None, :] +
                                                    want.abs())
    full = torch.empty((N, N), dtype=torch.float32, device="cuda")
    with torch.cuda.device(X.device):
        _lib.check(_lib.lib().skb_asnorm_apply(X.data_ptr(), N, D, mean.data_ptr(), std.data_ptr(), full.data_ptr(), _lib.stream_ptr()))
    assert excess(full, want, bound) <= 1.0
    for lo, hi in ((0, N), (137, 611)):
        panel = bulk._asnorm_panel_cuda(X, lo, hi, mean, std)
        assert excess(panel, want[lo:hi], bound[lo:hi]) <= 1.0, (lo, hi)


# ------------------------------------------------------------------------------------------------------------ PLDA
@pytest.mark.gpu
@pytest.mark.parametrize("D", (100, 150, 300))
def test_plda_scoring_against_the_oracle(D):
    """PLDA_scoring (skb_quadratic_prepare on the KC-64 / KC-128 / streamed kernels, then the score GEMM with passes=0)
    against the float64 oracle."""
    from oracle import scoring_ref as S
    Ne, Nt = 333, 517
    rng = numpy.random.default_rng(D)
    E, T = synth.synth_embeddings(Ne, D, seed=D + 1), synth.synth_embeddings(Nt, D, seed=D + 2)
    mu, F, Sigma = synth.synth_plda(D, D, seed=D + 3)
    ids_e = numpy.array(["m%d" % i for i in range(Ne)])
    ids_t = numpy.array(["s%d" % i for i in range(Nt)])
    ndx = sk.Ndx()
    ndx.modelset, ndx.segset = ids_e[rng.permutation(Ne)], ids_t[rng.permutation(Nt)]
    ndx.trialmask = rng.random((Ne, Nt)) < 0.5
    sc = sk.PLDA_scoring(sk.StatServer.from_embeddings(ids_e, E), sk.StatServer.from_embeddings(ids_t, T), ndx, mu, F,
                         numpy.zeros((D, 0)), Sigma)
    ref = S.fast_plda_scoring(ids_e, E, ids_t, T, ndx.modelset, ndx.segset, ndx.trialmask, mu, F, Sigma)
    assert numpy.array_equal(sc.modelset, ref[0]) and numpy.array_equal(sc.segset, ref[1])
    err = numpy.abs(sc.scoremat - ref[3])
    assert (err <= 2.5e-4 + 2e-6 * numpy.abs(ref[3])).all(), err.max()


# ------------------------------------------------------------------------------------------------- the pass rule
PASS_RULE_D = (64, 65, 100, 128, 200, 256, 512)


def pass_rule_error(D, same, n=20000, seed=81):
    """(max |S - ref|, S) for passes=0 on n x n unit-norm Gaussian rows (E = T when ``same``)."""
    E = operand("unit", n, D, seed)
    T = E if same else operand("unit", n, D, seed + 1)
    S = sk.score_matrix(E, T, passes=0)
    T64 = T.double()
    err = 0.0
    for i in range(0, n, 2000):
        err = max(err, (S[i:i + 2000].double() - E[i:i + 2000].double() @ T64.T).abs().max().item())
    return err, S, E, T


@pytest.mark.gpu
@pytest.mark.parametrize("same", (False, True))
@pytest.mark.parametrize("D", PASS_RULE_D)
def test_passes_0_keeps_its_error_promise_on_unit_rows(D, same):
    """passes=0 promises |S - E T^T| < 2.5e-4 for operands whose fp16 rounding errors are uncorrelated (20 000 x 20 000
    unit-norm Gaussian rows; E = T puts the squared norms, the largest errors, on the diagonal)."""
    err, _, _, _ = pass_rule_error(D, same)
    assert err < 2.5e-4, err


@pytest.mark.gpu
def test_unit_rows_of_width_256_and_512_stay_single_pass():
    for D in (256, 512):
        E, T = operand("unit", 300, D, 91), operand("unit", 200, D, 92)
        assert torch.equal(sk.score_matrix(E, T, passes=0), sk.score_matrix(E, T, passes=1)), D


@pytest.mark.gpu
@pytest.mark.parametrize("D", (100, 150, 200))
def test_three_passes_meet_their_bound_on_rows_of_one_repeated_value(D):
    """Coherent rounding: every entry of a row is the same value, so all fp16 rounding errors of a dot product share a
    sign.  No pass-count rule sees that; passes=3 is the bound."""
    E, T = operand("repeated", 2000, D, 101), operand("repeated", 3000, D, 102)
    out = sk.score_matrix(E, T, passes=3)
    ref, bound = reference(E, T, None, None, 0.0, 1.0, 3)
    assert excess(out, ref, bound) <= 1.0
    assert (out.double() - ref).abs().max().item() < 2.5e-4


# ------------------------------------------------------------------------------------------- operand checks
@pytest.mark.gpu
def test_a_column_slice_operand_is_scored_as_its_contiguous_copy():
    X = operand("gauss", 300, 256, 111)
    T = operand("gauss", 200, 200, 112)
    E = X[:, :200]
    want = sk.score_matrix(E.contiguous(), T, passes=3)
    assert torch.equal(sk.score_matrix(E, T, passes=3), want)
    assert torch.equal(sk.score_matrix(E.contiguous(), X[:200, :200], passes=3), sk.score_matrix(E.contiguous(), X[:200, :200].contiguous(), passes=3))
    mask = torch.rand((300, 200), generator=_gen(113), device="cuda") < 0.5
    assert torch.equal(score_trials(E, T, mask, passes=3), want[mask])
    vals, _ = sk.score_topk(E, T, 5, passes=3)
    assert torch.equal(vals, torch.sort(want, dim=1, descending=True).values[:, :5])
    r = torch.randn((600,), device="cuda")[::2]
    assert torch.equal(sk.score_matrix(E, T, r, passes=3), sk.score_matrix(E.contiguous(), T, r.contiguous(), passes=3))


@pytest.mark.gpu
def test_a_float64_operand_is_rejected():
    E = operand("gauss", 300, 128, 121).double()
    T = operand("gauss", 200, 128, 122)
    with pytest.raises(ValueError):
        sk.score_matrix(E, T)
    with pytest.raises(ValueError):
        sk.score_matrix(T, E)


@pytest.mark.gpu
def test_an_output_view_with_a_column_stride_is_rejected():
    E, T = operand("gauss", 300, 128, 131), operand("gauss", 200, 128, 132)
    buf = torch.zeros((300, 400), dtype=torch.float32, device="cuda")
    with pytest.raises(ValueError):
        sk.score_matrix(E, T, out=buf[:, ::2])


def _bad_calls(E, T, dev):
    """(name, thunk) pairs that must raise ValueError before any library call."""
    Ne, Nt = E.shape[0], T.shape[0]
    f32 = dict(dtype=torch.float32, device=dev)
    narrow = T[:, :-1].contiguous()
    calls = [
        ("T narrower than E", lambda: sk.score_matrix(E, narrow)),
        ("E narrower than T", lambda: sk.score_matrix(E[:, :-1], T)),
        ("1-D E", lambda: sk.score_matrix(E[0], T)),
        ("float16 T", lambda: sk.score_matrix(E, T.half())),
        ("rowterm too short", lambda: sk.score_matrix(E, T, torch.zeros((Ne - 1,), **f32))),
        ("colterm too long", lambda: sk.score_matrix(E, T, None, torch.zeros((Nt + 1,), **f32))),
        ("float64 colterm", lambda: sk.score_matrix(E, T, None, torch.zeros((Nt,), dtype=torch.float64, device=dev))),
        ("2-D rowterm", lambda: sk.score_matrix(E, T, torch.zeros((Ne, 1), **f32))),
        ("out too small", lambda: sk.score_matrix(E, T, out=torch.empty((Ne, Nt - 1), **f32))),
        ("out with too few rows", lambda: sk.score_matrix(E, T, out=torch.empty((Ne - 1, Nt), **f32))),
        ("int32 out", lambda: sk.score_matrix(E, T, out=torch.empty((Ne, Nt), dtype=torch.int32, device=dev))),
        ("out_dtype bfloat16", lambda: sk.score_matrix(E, T, out_dtype=torch.bfloat16)),
        ("trials, T narrower", lambda: score_trials(E, narrow, numpy.ones((Ne, Nt), bool))),
        ("trials, short colterm", lambda: score_trials(E, T, numpy.ones((Ne, Nt), bool), None, torch.zeros((Nt - 1,), **f32))),
        ("topk, T narrower", lambda: sk.score_topk(E, narrow, 2)),
        ("topk, short rowterm", lambda: sk.score_topk(E, T, 2, torch.zeros((Ne - 1,), **f32))),
    ]
    if dev.type == "cuda":
        cpu = torch.device("cpu")
        calls += [
            ("T on the host", lambda: sk.score_matrix(E, T.cpu())),
            ("out on the host", lambda: sk.score_matrix(E, T, out=torch.empty((Ne, Nt), dtype=torch.float32, device=cpu))),
            ("rowterm on the host", lambda: sk.score_matrix(E, T, torch.zeros((Ne,)))),
            ("packed T of another width", lambda: sk.score_matrix(E, PackedEmbeddings(narrow))),
            ("trials, packed T of another width", lambda: score_trials(E, PackedEmbeddings(narrow), numpy.ones((Ne, Nt), bool))),
            ("topk, packed T of another width", lambda: sk.score_topk(E, PackedEmbeddings(narrow), 2)),
        ]
    return calls


def test_host_operands_are_rejected_before_any_library_call():
    E, T = torch.randn((30, 16)), torch.randn((20, 16))
    for name, call in _bad_calls(E, T, torch.device("cpu")):
        with pytest.raises(ValueError):
            call()
            pytest.fail(name)


@pytest.mark.gpu
def test_malformed_device_operands_are_rejected_before_any_library_call():
    E, T = operand("gauss", 30, 16, 141), operand("gauss", 20, 16, 142)
    for name, call in _bad_calls(E, T, E.device):
        with pytest.raises(ValueError):
            call()
            pytest.fail(name)
