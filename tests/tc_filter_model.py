"""numpy model of the tensor-core tokeniser's candidate FILTER (csrc/rq_tcx.cu) -- test infrastructure.

The kernel's exactness argument has two halves: the exact fp32 re-rank (same arithmetic as the CUDA-core kernel, tested
against the oracle on the GPU) and the claim that the fp16 tensor-core scores never drop the true argmin from the candidate
set {k : h[k] <= min h + 2 eps_b}.  The second half is a DETERMINISTIC bound (DESIGN.md 5.2 "filter error bound") and this
model restates it on the CPU with the kernel's own formulas, so the margin can be checked -- and changed -- without a GPU:

  x~ = fp16(x), c~ = fp16(c * 2^s) / 2^s        (tc_prep_blob_kernel, converter; the power-of-two scale is exact)
  S  = x~ . c~                                  (tcgen05.mma, fp32 accumulation)
  h  = T[k] - S,  T = cc/2 + sum_j G_jl[id_j]   (Gram tables from float64, rounded once; epilogue)
  x~.c~ - x.c = (x~ - x).c~ + x.(c~ - c)   exactly, so by Cauchy-Schwarz
  |x~.c~ - x.c| <= ||x~ - x|| ||c~_k|| + ||x|| ||c~_k - c_k||  <=  ex_b chat_l + xn_b ec_l
     ex_b = ||x~ - x||_2 MEASURED per row by the converter (covers subnormals / flushes / overflow by itself),
     chat_l = max_k ||c~_k||, ec_l = max_k ||c~_k - c_k|| measured by tc_prep_err_kernel
  eps_b = 1.002 (ex_b chat_l + xn_b ec_l) + 2^-17 xn_b c2max_l (tensor-core accumulation, 64 ulp of the partial-sum bound)
          + gerr_l (Gram / table / FFMA roundings) + ref_l(b) (fp32 evaluation noise of the REFERENCE's own distances)
  candidates = {k : h[k] <= min h + 2 eps_b (1 + 2^-16)}
"""
import numpy as np

U16 = 2.0 ** -11
INFL = 1.002          # fp32 accumulation of the measured norms + bf16 round-up of the row statistics are inside this


def _bf16_up(v):
    b = np.asarray(v, np.float32).view(np.uint32).copy()
    fin = (b & 0x7F800000) != 0x7F800000
    b[fin & ((b & 0xFFFF) != 0)] += 0x10000
    return (b & 0xFFFF0000).view(np.float32)


def prepare(cbs):
    """Per-level constants of tc_prep_stats_kernel / tc_prep_consts_kernel / tc_prep_err_kernel and the fp16 images."""
    lv = []
    for l, c in enumerate(cbs):
        c = np.asarray(c, np.float32)
        amax = float(np.abs(c).max())
        sc = 1.0
        if amax > 0 and np.isfinite(amax):
            e = int(np.clip(np.frexp(amax)[1], -60, 60))
            sc = float(np.ldexp(1.0, -e))
        c64 = c.astype(np.float64)
        with np.errstate(over="ignore"):
            img = (c * np.float32(sc)).astype(np.float16)
        ct = img.astype(np.float64) / sc                      # c~ as real numbers
        lv.append(dict(sc=sc, c2max=float(np.sqrt((c64 ** 2).sum(1)).max()),
                       chat=float(np.sqrt((ct ** 2).sum(1)).max()) * INFL,
                       ec=float(np.sqrt(((ct - c64) ** 2).sum(1)).max()) * INFL,
                       cc=(c64 * c64).sum(1), img=img))
    for l in range(len(cbs)):
        prior = sum(lv[j]["c2max"] for j in range(l))
        lv[l]["prior"] = prior
        lv[l]["gerr"] = 2.0 ** -22 * (lv[l]["c2max"] * prior + 0.5 * lv[l]["c2max"] ** 2)
    return lv


def gram_tables(cbs):
    """G[(j, l)] = C_j C_l^T from float64, rounded to fp32 once (tc_prep_gram_kernel); cc_l / 2 folded into j = 0."""
    out = {}
    for l in range(1, len(cbs)):
        cl = np.asarray(cbs[l], np.float64)
        for j in range(l):
            g = np.asarray(cbs[j], np.float64) @ cl.T
            if j == 0:
                g = g + 0.5 * (cl * cl).sum(1)[None, :]
            out[(j, l)] = g.astype(np.float32)
    return out


def row_stats(x):
    """(ex^2, xn^2) as the converter publishes them: fp32 sums, bf16 rounded up."""
    x = np.asarray(x, np.float32)
    with np.errstate(over="ignore", invalid="ignore"):
        xh = x.astype(np.float16)
        d = xh.astype(np.float64) - x.astype(np.float64)
        ex2 = _bf16_up((d * d).sum(1).astype(np.float32))
        xn2 = _bf16_up((x.astype(np.float64) ** 2).sum(1).astype(np.float32))
    return xh, ex2, xn2


def eps_of(lvl, ex2, xn2):
    ex = np.sqrt(ex2.astype(np.float64))
    xn = np.sqrt(xn2.astype(np.float64))
    acc = 2.0 ** -17 * xn * lvl["c2max"]
    ref = 2.0 ** -17 * ((xn + lvl["prior"]) * lvl["c2max"] + 0.5 * lvl["c2max"] ** 2)
    return INFL * (ex * lvl["chat"] + xn * lvl["ec"]) + acc + lvl["gerr"] + ref


def filter_levels(x, cbs, ids):
    """ids: the exact chain's ids [B, L] (the kernel feeds the FINAL ids of earlier levels into the Gram correction).
    Returns per level: candidate mask [B, K], eps [B], approximate half-distances h [B, K]."""
    x = np.asarray(x, np.float32)
    B, D = x.shape
    lv = prepare(cbs)
    grams = gram_tables(cbs)
    xh, ex2, xn2 = row_stats(x)
    out = []
    for l, c in enumerate(cbs):
        k = lv[l]
        with np.errstate(over="ignore", invalid="ignore"):
            S = (xh.astype(np.float64) @ k["img"].astype(np.float64).T).astype(np.float32)
        if l == 0:
            T = np.broadcast_to((0.5 * k["cc"]).astype(np.float32), (B, len(k["cc"]))).copy()
        else:
            T = grams[(0, l)][ids[:, 0]].copy()
            for j in range(1, l):
                T += grams[(j, l)][ids[:, j]]
        with np.errstate(over="ignore", invalid="ignore"):
            h = (T - S * np.float32(1.0 / k["sc"])).astype(np.float32)
            eps = eps_of(k, ex2, xn2)
            m1 = np.nanmin(np.where(np.isnan(h), np.inf, h), axis=1)
            thr = m1 + 2.0 * eps * (1 + 2.0 ** -16)
            cand = ~(h > thr[:, None])
        out.append(dict(cand=cand, eps=eps, h=h))
    return out


def true_half_distances(x, cbs, ids, level):
    """float64 half-distance cc/2 - res.c of `level` along the chain given by ids."""
    res = np.asarray(x, np.float64).copy()
    for j in range(level):
        res -= np.asarray(cbs[j], np.float64)[ids[:, j]]
    c = np.asarray(cbs[level], np.float64)
    return 0.5 * (c * c).sum(1)[None, :] - res @ c.T


# ---- adversarial inputs: structured rounding errors that defeat a statistical (z sigma) margin ----------------------
def adversarial_problem(kind: str, D: int = 768, K: int = 256, L: int = 1, n: int = 64, seed: int = 5):
    """Rows / codebooks whose fp16 rounding errors are coherent (same sign, parallel to a code).  Returns (x, cbs)."""
    rs = np.random.RandomState(seed)
    s = np.where(rs.rand(D) < 0.5, -1.0, 1.0)
    if kind == "judge_r1":
        # VERDICT round 1, weak point 1: every element of x rounds DOWN to 2^-5 in fp16 (same-signed error), two codes
        # parallel to x whose true gap (1.9e-3 relative) is smaller than the coherent error but 200x the near-tie tau
        x = np.tile((s * 2.0 ** -5 * (1 + 0.99 * 2.0 ** -11)).astype(np.float32), (n, 1))
        cb = (1e-3 * rs.randn(K, D)).astype(np.float32)
        cb[10] = (0.046875 * s).astype(np.float32)
        cb[200] = ((0.015625 + 2.0 ** -16) * s).astype(np.float32)
        cbs = [cb] + [(1e-3 * rs.randn(K, D)).astype(np.float32) for _ in range(L - 1)]
        return x, cbs
    if kind == "sign_biased":
        # unit-norm rows whose mantissas sit just below a rounding boundary (all round up), correlated with half the codes
        base = rs.randn(n, D)
        base /= np.sqrt((base ** 2).sum(1, keepdims=True))
        h = base.astype(np.float16).astype(np.float64)
        ulp = np.abs(np.spacing(h.astype(np.float16)).astype(np.float64))
        x = (h + np.sign(h) * 0.49 * ulp).astype(np.float32)        # fp16 rounds every element toward zero by ~ulp/2
        cbs = []
        res = x.astype(np.float64)
        for _ in range(L):
            idx = rs.choice(n, K, replace=True)
            cb = res[idx] * (1 + 0.002 * rs.randn(K, 1)) + 1e-4 * rs.randn(K, D)
            cb = cb.astype(np.float32)
            cbs.append(cb)
            d = (cb.astype(np.float64) ** 2).sum(1)[None] - 2 * res @ cb.astype(np.float64).T
            res = res - cb.astype(np.float64)[d.argmin(1)]
        return x, cbs
    if kind == "equal_magnitude":
        # |x_d| identical everywhere (one fp16 binade, identical relative error), codes = +-1 patterns at nearby scales
        v = 0.03 * (1 + 0.37 * 2.0 ** -11)
        x = (np.where(rs.rand(n, D) < 0.5, -1.0, 1.0) * v).astype(np.float32)
        cbs = []
        for _ in range(L):
            idx = rs.choice(n, K, replace=True)
            scale = 1 + 2.0 ** -9 * rs.randint(-8, 9, size=(K, 1))
            cbs.append((x[idx] * scale).astype(np.float32))
        return x, cbs
    if kind == "code_parallel":
        # codes are exact multiples of a few rows: many near-parallel candidates with tiny true gaps at several scales
        base = rs.randn(8, D)
        base /= np.sqrt((base ** 2).sum(1, keepdims=True))
        x = (base[rs.randint(0, 8, n)] * (1 + 1e-3 * rs.randn(n, 1))).astype(np.float32)
        cbs = []
        for _ in range(L):
            cb = base[rs.randint(0, 8, K)] * (1 + 3e-4 * rs.randn(K, 1))
            cbs.append(cb.astype(np.float32))
        return x, cbs
    if kind == "opposite_rounding":
        # x exact in fp16 (ex = 0) and, per row, two codes parallel to it whose fp16 roundings go opposite ways by 0.49 ulp per
        # element: the scores move the truly closer code B up and the other code A down by ~eps each, so B stays a candidate
        # only under the full 2 eps margin (B - A is 1.5e-4 in half-distance: far above fp32 noise and the near-tie tolerance).
        # Row i follows sign pattern p = i % 64 with codes p and 128 + p, one in each CTA's half of the 256 codes; which of the
        # two is B alternates with p.
        a, ulp = 0.046875, 2.0 ** -15                  # 1.5 * 2^-5 is exact in fp16; ulp of its binade
        pats = np.where(rs.rand(64, D) < 0.5, -1.0, 1.0)
        x = (pats[np.arange(n) % 64] * a).astype(np.float32)
        cb = (1e-3 * rs.randn(K, D)).astype(np.float32)
        for p in range(64):
            ib, ia = (p, 128 + p) if p % 2 == 0 else (128 + p, p)
            cb[ib] = pats[p] * (a + 0.49 * ulp)        # rounds down to a
            cb[ia] = pats[p] * (a - 20.49 * ulp)       # rounds up to a - 20 ulp
        cbs = [cb] + [(1e-3 * rs.randn(K, D)).astype(np.float32) for _ in range(L - 1)]
        return x, cbs
    if kind == "tiny_and_huge":
        # rows spanning fp16 subnormal .. overflow scales
        base = rs.randn(n, D)
        base /= np.sqrt((base ** 2).sum(1, keepdims=True))
        scale = 10.0 ** rs.uniform(-7, 5.5, size=(n, 1))
        x = (base * scale).astype(np.float32)
        cbs = [(base[rs.choice(n, K, replace=True)] * 10.0 ** rs.uniform(-2, 1, size=(K, 1))
                + 1e-3 * rs.randn(K, D)).astype(np.float32) for _ in range(L)]
        return x, cbs
    raise ValueError(kind)


ADVERSARIAL_KINDS = ["judge_r1", "sign_biased", "equal_magnitude", "code_parallel", "tiny_and_huge", "opposite_rounding"]
