"""GPU parity tests proper: the CUDA path (through the C ABI) against the oracle on seeded inputs and against
the committed reference-generated fixtures.  Run with `pytest -m gpu` on a B200."""
import numpy as np
import pytest
import torch

import inputs as I
from oracle import rq_oracle as O
from parity import assert_ids_match, load_golden, rel_err

pytestmark = pytest.mark.gpu

T, BETA = 0.2, 0.25
TOL = 1e-5
KMODE = {"eval": 0, "ste": 2, "rot": 3}
OMODE = {"eval": O.STE, "ste": O.STE, "rot": O.ROTATION_TRICK, "gumbel": O.GUMBEL_SOFTMAX}


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.detach().cpu().numpy()


@pytest.fixture(scope="module")
def ops():
    from rq_vae_recommender_b200 import ops as _ops
    return _ops


# ------------------------------------------------------------------ fused chain vs golden (reference outputs)
@pytest.mark.parametrize("tag", ["c1", "d32", "d768"])
@pytest.mark.parametrize("mname", ["eval", "ste", "rot"])
def test_single_level_vs_reference(ops, tag, mname):
    g = load_golden("quantize_levels")
    B, D, K, keep = (int(v) for v in g[f"{tag}_shape"])
    x, cbs = I.rq_problem(B, D, K, 1, seed=100 + D)
    o = ops.rq_forward(dev(x), [dev(cbs[0])], KMODE[mname], BETA, want_ids=True, want_embeddings=True,
                       want_residuals=True, want_sum=True, want_norms=True, want_loss=True)
    ids = host(o["ids"])[:, 0]
    ref_ids = g[f"{tag}_{mname}_ids"].astype(np.int64)
    assert_ids_match(ids, ref_ids, x, cbs, f"{tag}/{mname}")
    same = ids == ref_ids
    assert same.mean() > 0.999
    assert rel_err(host(o["loss"])[same], g[f"{tag}_{mname}_loss"][same]) < TOL
    emb = host(o["embeddings"])[0]
    assert rel_err(emb[:keep][same[:keep]], g[f"{tag}_{mname}_emb"][same[:keep]]) < 2e-5
    assert rel_err(emb.astype(np.float64).sum(1)[same], g[f"{tag}_{mname}_emb_rowsum"][same]) < 2e-5
    assert np.array_equal(host(o["residuals"])[0], x)
    assert np.array_equal(host(o["emb_sum"]), emb)
    assert rel_err(host(o["emb_norms"])[:, 0], np.sqrt((emb.astype(np.float64) ** 2).sum(1))) < TOL


@pytest.mark.parametrize("mname", ["eval", "ste", "rot"])
def test_ns_chain_vs_reference(ops, mname):
    g = load_golden("rq_ns2048")
    n, D, K, L = (int(v) for v in g["shape"])
    x, cbs = I.rq_problem(n, D, K, L, seed=1234)
    o = ops.rq_forward(dev(x), [dev(c) for c in cbs], KMODE[mname], BETA, want_ids=True, want_sum=True,
                       want_norms=True, want_loss=True)
    ids = host(o["ids"])
    n_tie = assert_ids_match(ids, g[f"{mname}_ids"], x, cbs, mname)
    same = (ids == g[f"{mname}_ids"]).all(1)
    assert n_tie <= 2
    assert rel_err(host(o["loss"])[same], g[f"{mname}_loss"][same]) < TOL
    assert rel_err(host(o["emb_norms"])[same], g[f"{mname}_embs_norm"][same]) < TOL
    assert np.abs(host(o["emb_sum"])[:32] - g[f"{mname}_embsum_head"])[same[:32]].max() < 1e-6


def test_beauty_codebooks_vs_reference(ops):
    g = load_golden("beauty_ckpt")
    cbs = list(g["codebooks"])
    o = ops.rq_forward(dev(g["res"]), [dev(c) for c in cbs], 0, BETA, want_ids=True, want_norms=True, want_loss=True)
    ids = host(o["ids"])
    n_tie = assert_ids_match(ids, g["sem_ids"], g["res"], cbs)
    same = (ids == g["sem_ids"]).all(1)
    assert n_tie <= 4
    assert rel_err(host(o["loss"])[same], g["qloss"][same]) < TOL
    assert rel_err(host(o["emb_norms"])[same], g["embs_norm"][same]) < TOL


# ------------------------------------------------------------------ fused chain vs oracle: ragged / edge shapes
@pytest.mark.parametrize("B,D,K,L", [(1, 16, 32, 2), (7, 20, 5, 3), (333, 64, 256, 3), (1000, 36, 300, 2),
                                      (129, 128, 100, 4), (65, 768, 256, 3), (40, 1536, 64, 2)])
@pytest.mark.parametrize("mname", ["eval", "ste", "rot"])
def test_chain_vs_oracle_shapes(ops, B, D, K, L, mname):
    x, cbs = I.rq_problem(max(B, K), D, K, L, seed=B + D)
    x = x[:B]
    so = O.rq_forward(x, cbs, OMODE[mname], mname != "eval", T, BETA)
    o = ops.rq_forward(dev(x), [dev(c) for c in cbs], KMODE[mname], BETA, want_ids=True, want_embeddings=True,
                       want_residuals=True, want_sum=True, want_norms=True, want_loss=True)
    ids = host(o["ids"])
    assert_ids_match(ids, so.sem_ids, x, cbs)
    same = (ids == so.sem_ids).all(1)
    assert same.mean() > 0.98
    emb = host(o["embeddings"]).transpose(1, 2, 0)
    res = host(o["residuals"]).transpose(1, 2, 0)
    assert rel_err(emb[same], so.embeddings[same]) < 2e-5
    assert np.abs(res[same] - so.residuals[same]).max() < 1e-5
    assert rel_err(host(o["loss"])[same], so.quantize_loss[same]) < 2e-5
    assert rel_err(host(o["emb_sum"])[same], so.embeddings.sum(-1)[same]) < 2e-5


def test_empty_and_strided_inputs(ops):
    cb = dev(I.randn(1, 32, 16))
    o = ops.rq_forward(torch.empty(0, 16, device="cuda"), [cb], 0, BETA, want_ids=True, want_loss=True)
    assert o["ids"].shape == (0, 1) and o["loss"].shape == (0,)
    x = I.randn(2, 50, 40)
    xs = dev(x)[:, 4:20]                       # row stride 40, width 16, offset 4 floats (16B aligned)
    a = host(ops.rq_tokenize(xs, [cb]))
    b = host(ops.rq_tokenize(xs.contiguous(), [cb]))
    assert np.array_equal(a, b)
    xs2 = dev(x)[:, 3:19]                      # misaligned start -> scalar load path
    assert np.array_equal(host(ops.rq_tokenize(xs2, [cb])), host(ops.rq_tokenize(xs2.contiguous(), [cb])))


def test_exact_ties_pick_first_index(ops):
    cb = I.randn(3, 32, 16)
    cb[17] = cb[5]
    cb[30] = cb[5]
    x = np.repeat(cb[5:6], 64, axis=0) + 1e-3 * I.randn(4, 64, 16)
    ids = host(ops.rq_tokenize(dev(x), [dev(cb)]))[:, 0]
    assert (ids == 5).all()


# ------------------------------------------------------------------ backward vs reference autograd (golden) and oracle
@pytest.mark.parametrize("tag", ["c1", "d32", "d768"])
@pytest.mark.parametrize("mname", ["ste", "rot"])
def test_single_level_backward_vs_reference(ops, tag, mname):
    g = load_golden("quantize_levels")
    B, D, K, keep = (int(v) for v in g[f"{tag}_shape"])
    x, cbs = I.rq_problem(B, D, K, 1, seed=100 + D)
    g_out, g_loss = I.randn(200 + D, B, D), I.rand(201 + D, B)
    xt = dev(x).requires_grad_(True)
    ct = dev(cbs[0]).requires_grad_(True)
    embs, _res, ids, loss = ops.RqChainFunction.apply(xt, KMODE[mname], BETA, False, ct)
    ((embs[0] * dev(g_out)).sum() + (loss * dev(g_loss)).sum()).backward()
    same = host(ids)[:, 0] == g[f"{tag}_{mname}_ids"]
    assert same.mean() > 0.999
    gx = host(xt.grad)
    assert rel_err(gx[:keep][same[:keep]], g[f"{tag}_{mname}_gx"][same[:keep]]) < 2e-5
    if same.all():
        assert rel_err(gx.astype(np.float64).sum(1), g[f"{tag}_{mname}_gx_rowsum"]) < 2e-5
        gc = host(ct.grad)
        assert rel_err(gc if D <= 32 else gc[:, :32], g[f"{tag}_{mname}_gc"]) < 2e-5
        assert rel_err(gc.astype(np.float64).sum(1), g[f"{tag}_{mname}_gc_rowsum"]) < 2e-5


@pytest.mark.parametrize("mname", ["eval", "ste", "rot"])
@pytest.mark.parametrize("lean", [False, True])
def test_chain_backward_vs_torch_autograd_of_oracle_formulas(ops, mname, lean):
    """Multi-level chain gradient: compare with float64 torch autograd of the reference expressions."""
    B, D, K, L = 257, 24, 40, 3
    x, cbs = I.rq_problem(max(B, K), D, K, L, seed=5)
    x = x[:B]
    xt = dev(x).requires_grad_(True)
    cts = [dev(c).requires_grad_(True) for c in cbs]
    a, b, ids, loss = ops.RqChainFunction.apply(xt, KMODE[mname], BETA, lean, *cts)
    ga = dev(I.randn(11, *a.shape))
    gb = dev(I.randn(12, *b.shape))
    gl = dev(I.rand(13, B))
    obj = (a * ga).sum() + (loss * gl).sum()
    if not lean:
        obj = obj + (b * gb).sum()
    obj.backward()
    # float64 reference on the SAME ids
    ids_h = ids.cpu()
    x64 = torch.from_numpy(x).double().requires_grad_(True)
    c64 = [torch.from_numpy(c).double().requires_grad_(True) for c in cbs]
    res = x64
    embs, ress, tot = [], [], 0
    for l in range(L):
        ress.append(res)
        e = c64[l][ids_h[:, l]]
        if mname == "eval":
            eo = e
        elif mname == "ste":
            eo = res + (e - res).detach()
        else:
            u = res / (res.norm(dim=-1, keepdim=True) + 1e-8)
            q = e / (e.norm(dim=-1, keepdim=True) + 1e-8)
            w = torch.nn.functional.normalize(u + q, p=2, dim=1, eps=1e-6).detach()
            rot = res - 2 * (res * w).sum(1, keepdim=True) * w + 2 * (res * u.detach()).sum(1, keepdim=True) * q.detach()
            eo = rot * (e.norm(dim=1, keepdim=True) / (res.norm(dim=1, keepdim=True) + 1e-6)).detach()
        tot = tot + ((res.detach() - e) ** 2).sum(-1) + BETA * ((res - e.detach()) ** 2).sum(-1)
        res = res - eo
        embs.append(eo)
    E = torch.stack(embs, 0)
    if lean:
        obj64 = (E.sum(0) * ga.cpu().double()).sum() + (tot * gl.cpu().double()).sum()
    else:
        obj64 = (E * ga.cpu().double()).sum() + (torch.stack(ress, 0) * gb.cpu().double()).sum() + (tot * gl.cpu().double()).sum()
    obj64.backward()
    assert rel_err(host(xt.grad), x64.grad.numpy()) < 2e-5
    for ct, c in zip(cts, c64):
        assert rel_err(host(ct.grad), c.grad.numpy()) < 2e-5


# ------------------------------------------------------------------ Gumbel level
@pytest.mark.parametrize("tag", ["c1", "d32", "d768"])
def test_gumbel_level_vs_reference(ops, tag):
    g = load_golden("quantize_levels")
    B, D, K, keep = (int(v) for v in g[f"{tag}_shape"])
    x, cbs = I.rq_problem(B, D, K, 1, seed=100 + D)
    g_out, g_loss, u = I.randn(200 + D, B, D), I.rand(201 + D, B), I.rand(202 + D, B, K)
    xt = dev(x).requires_grad_(True)
    ct = dev(cbs[0]).requires_grad_(True)
    emb, ids, loss = ops.GumbelQuantizeFunction.apply(xt, ct, dev(u), T, BETA)
    ((emb * dev(g_out)).sum() + (loss * dev(g_loss)).sum()).backward()
    assert_ids_match(host(ids), g[f"{tag}_gumbel_ids"], x, cbs)
    # softmax at T=0.2 amplifies fp32 rounding of dist by 1/T: compare at 5e-4 like the oracle test
    assert rel_err(host(loss), g[f"{tag}_gumbel_loss"]) < 5e-4
    assert rel_err(host(emb)[:keep], g[f"{tag}_gumbel_emb"]) < 5e-4
    assert rel_err(host(emb).astype(np.float64).sum(1), g[f"{tag}_gumbel_emb_rowsum"]) < 5e-4
    gx, gc = host(xt.grad), host(ct.grad)
    assert rel_err(gx[:keep], g[f"{tag}_gumbel_gx"]) < 1e-3
    assert rel_err(gc if D <= 32 else gc[:, :32], g[f"{tag}_gumbel_gc"]) < 1e-3
    assert rel_err(gc.astype(np.float64).sum(1), g[f"{tag}_gumbel_gc_rowsum"]) < 1e-3


# ------------------------------------------------------------------ dense helpers
@pytest.mark.parametrize("M,N,K", [(1, 1, 1), (130, 70, 33), (256, 512, 768), (1000, 32, 128)])
@pytest.mark.parametrize("ta,tb", [(False, False), (False, True), (True, False), (True, True)])
def test_sgemm(ops, M, N, K, ta, tb):
    a = I.randn(1, *((K, M) if ta else (M, K)))
    b = I.randn(2, *((N, K) if tb else (K, N)))
    ref = (a.T if ta else a).astype(np.float64) @ (b.T if tb else b).astype(np.float64)
    out = host(ops.sgemm(dev(a), dev(b), trans_a=ta, trans_b=tb))
    assert rel_err(out, ref) < 1e-5
    out = host(ops.sgemm(dev(a), dev(b), trans_a=ta, trans_b=tb, relu=True))
    assert rel_err(out, np.maximum(ref, 0)) < 1e-5


def test_mlp_vs_reference(ops):
    g = load_golden("mlp")
    ws = I.mlp_weights(500, [768, 512, 256, 128, 32])
    x = I.unit_rows(501, 256, 768)
    gy = I.randn(502, 256, 32)
    for norm in (False, True):
        xt = dev(x).requires_grad_(True)
        wts = [dev(w).requires_grad_(True) for w in ws]
        y = ops.MLPFunction.apply(xt, norm, *wts)
        (y * dev(gy)).sum().backward()
        assert rel_err(host(y), g[f"y_norm{int(norm)}"]) < TOL
        gx, gx_ref = host(xt.grad), g[f"gx_norm{int(norm)}"]           # the fixture keeps the first rows of gx
        assert rel_err(gx[:len(gx_ref)], gx_ref) < 2e-5
        assert rel_err(gx.astype(np.float64).sum(1), g[f"gx_rowsum_norm{int(norm)}"]) < 2e-5
        assert rel_err(host(wts[3].grad), g[f"gw3_norm{int(norm)}"]) < 2e-5
        assert rel_err(host(wts[0].grad).astype(np.float64).sum(1), g[f"gw0_rowsum_norm{int(norm)}"]) < 2e-5
    assert rel_err(host(ops.l2norm_rows(dev(I.randn(503, 256, 40)))), g["l2norm"]) < TOL


# ------------------------------------------------------------------ k-means
@pytest.mark.parametrize("tag,k,iters", [("a", 32, None), ("b", 256, 6), ("dup", 32, 4)])
def test_kmeans_vs_reference(tag, k, iters):
    from rq_vae_recommender_b200.init import kmeans as KM
    g = load_golden("kmeans")
    x = {"a": lambda: I.randn(600, 4096, 16), "b": lambda: I.randn(601, 20000, 32),
         "dup": lambda: np.repeat(np.round(I.randn(602, 24, 8) * 8) / 8, 16, axis=0)}[tag]()
    np.random.seed(610)
    torch.manual_seed(611)
    km = KM.Kmeans(k=k, max_iters=iters)
    out = km.run(dev(x))
    agree = (host(out.assignment) == g[f"{tag}_assignment"]).mean()
    assert agree > 0.999, agree
    assert np.abs(host(out.centroids) - g[f"{tag}_centroids"]).max() < 2e-5
    if tag == "a":
        w = torch.zeros(32, 16, device="cuda")
        np.random.seed(610)
        KM.kmeans_init_(w, dev(x))
        assert np.abs(host(w) - g["a_centroids"]).max() < 2e-5


def test_sid_histogram(ops):
    ids = np.random.RandomState(3).randint(0, 256, size=(5000, 3)).astype(np.int64)
    h = host(ops.sid_histogram(dev(ids), 256))
    assert np.array_equal(h, O.codebook_usage(ids, 256))


# ------------------------------------------------------------------ bf16 tensor-core MLP (reduced precision, opt-in)
@pytest.mark.parametrize("M,dims", [(1, [64, 64]), (130, [128, 64, 32]), (1000, [768, 512, 256, 128, 32]),
                                     (257, [192, 320, 70])])
def test_gemm_bf16_mlp_vs_bf16_oracle(ops, M, dims):
    """tcgen05 bf16 GEMM chain vs the oracle's bf16-rounding emulation of the reference under autocast."""
    x = I.randn(40, M, dims[0]) * 0.3
    ws = I.mlp_weights(41, dims)
    dws = [dev(w) for w in ws]
    # (1) TIGHT, layer by layer.  The kernel's fp32 output of the first k layers (pre-activation of layer k) is what its
    #     own epilogue rounds to bf16 for layer k+1, so feeding round_bf16(relu(.)) of it to the oracle removes the only
    #     legitimate source of large differences (an activation landing on the other side of a bf16 rounding boundary):
    #     what is left is fp32-vs-float64 accumulation order.
    prev = None
    for k in range(1, len(ws) + 1):
        yk = host(ops.mlp_forward_bf16(dev(x), dws[:k]))
        h = O.round_bf16(x) if prev is None else O.round_bf16(np.maximum(prev, 0))
        expect = h.astype(np.float64) @ O.round_bf16(ws[k - 1]).astype(np.float64).T
        assert yk.shape == (M, dims[k])
        assert rel_err(yk, expect) < 1e-5, (k, rel_err(yk, expect))
        prev = yk
    # (2) END TO END against the pure oracle chain.  Here a few intermediate activations legitimately round the other
    #     way (fp32-in-TMEM vs float64 accumulation on opposite sides of a bf16 boundary, 1 ulp = 0.4 %); measured on
    #     the 4-layer shipped architecture: most outputs bit-identical, ~1/4 of rows touched at a few 1e-4, max 2.6e-3.
    #     (1) above is the correctness proof; this bounds the bulk tightly and the tail by a few bf16 ulps.
    for norm in (False, True):
        y = host(ops.mlp_forward_bf16(dev(x), dws, normalize=norm))
        ref = O.mlp_forward_bf16(x, ws, normalize=norm)
        assert y.shape == ref.shape == (M, dims[-1])
        err = np.abs(y.astype(np.float64) - ref) / np.abs(ref).max()
        stats = (np.median(err), np.quantile(err, 0.99), err.max())
        assert stats[0] < 1e-6 and stats[1] < 2e-3 and stats[2] < 1e-2, stats
    # and it is the reduced-precision path: close to, but not equal to, the exact fp32 MLP
    exact = O.mlp_forward(x, ws)
    y = host(ops.mlp_forward_bf16(dev(x), dws))
    assert 1e-5 < rel_err(y, exact) < 5e-2


def test_gemm_bf16_single_layer_exact_products(ops):
    """One layer, inputs already representable in bf16: products are exact, only fp32 accumulation order differs."""
    M, K, N = 300, 256, 512
    x = O.round_bf16(I.randn(42, M, K))
    w = O.round_bf16(I.randn(43, N, K) * 0.1)
    y = host(ops.mlp_forward_bf16(dev(x), [dev(w)]))
    ref = x.astype(np.float64) @ w.astype(np.float64).T
    assert rel_err(y, ref) < 1e-5
    with pytest.raises(Exception):
        ops.mlp_forward_bf16(dev(I.randn(1, 8, 100)), [dev(I.randn(2, 16, 100))])     # K not a multiple of 64
