"""Pins the numpy oracle (oracle/rq_oracle.py) against outputs of the UNMODIFIED reference
(tests/golden/*.npz, written by tests/golden/make_golden.py in the build container).  CPU only."""
import numpy as np
import pytest

import inputs as I
from oracle import rq_oracle as O
from parity import assert_ids_match, load_golden, rel_err

T, BETA = 0.2, 0.25
MODE = {"ste": O.STE, "rot": O.ROTATION_TRICK, "gumbel": O.GUMBEL_SOFTMAX}
TOL = 1e-5


def _quantize_inputs(tag, g):
    B, D, K, keep = (int(v) for v in g[f"{tag}_shape"])
    x, cbs = I.rq_problem(B, D, K, 1, seed=100 + D)
    g_out, g_loss, u = I.randn(200 + D, B, D), I.rand(201 + D, B), I.rand(202 + D, B, K)
    assert I.sha(x, cbs[0], g_out, g_loss, u) == str(g[f"{tag}_sha"]), "regenerated inputs differ from the fixture"
    return x, cbs[0], g_out, g_loss, u, keep


@pytest.mark.parametrize("tag", ["c1", "d32", "d768"])
def test_quantize_eval(tag):
    g = load_golden("quantize_levels")
    x, cb, *_, keep = _quantize_inputs(tag, g)
    o = O.quantize_forward(x, cb, training=False, beta=BETA)
    assert_ids_match(o.ids, g[f"{tag}_eval_ids"], x, [cb], tag)
    same = o.ids == g[f"{tag}_eval_ids"]
    assert rel_err(o.loss[same], g[f"{tag}_eval_loss"][same]) < TOL
    assert rel_err(o.embeddings[:keep][same[:keep]], g[f"{tag}_eval_emb"][same[:keep]]) < TOL
    assert rel_err(o.embeddings.astype(np.float64).sum(1)[same], g[f"{tag}_eval_emb_rowsum"][same]) < TOL


@pytest.mark.parametrize("tag", ["c1", "d32", "d768"])
@pytest.mark.parametrize("mname", ["ste", "rot", "gumbel"])
def test_quantize_train_fwd_bwd(tag, mname):
    g = load_golden("quantize_levels")
    x, cb, g_out, g_loss, u, keep = _quantize_inputs(tag, g)
    o = O.quantize_forward(x, cb, MODE[mname], True, T, BETA, u)
    assert_ids_match(o.ids, g[f"{tag}_{mname}_ids"], x, [cb], tag)
    same = o.ids == g[f"{tag}_{mname}_ids"]
    assert same.mean() > 0.999
    assert rel_err(o.loss[same], g[f"{tag}_{mname}_loss"][same]) < TOL
    assert rel_err(o.embeddings[:keep][same[:keep]], g[f"{tag}_{mname}_emb"][same[:keep]]) < 2e-5
    assert rel_err(o.embeddings.astype(np.float64).sum(1)[same], g[f"{tag}_{mname}_emb_rowsum"][same]) < 2e-5
    gx, gc = O.quantize_backward(MODE[mname], x, cb, g[f"{tag}_{mname}_ids"].astype(np.int64), g_out, g_loss,
                                 BETA, T, u)
    # the gumbel softmax at T=0.2 amplifies fp32 rounding of dist by 1/T before exp(): looser there
    tol = 5e-4 if mname == "gumbel" else 2e-5
    assert rel_err(gx[:keep], g[f"{tag}_{mname}_gx"]) < tol
    assert rel_err(gx.astype(np.float64).sum(1), g[f"{tag}_{mname}_gx_rowsum"]) < tol
    D = cb.shape[1]
    assert rel_err(gc if D <= 32 else gc[:, :32], g[f"{tag}_{mname}_gc"]) < tol
    assert rel_err(gc.astype(np.float64).sum(1), g[f"{tag}_{mname}_gc_rowsum"]) < tol


def _c1(n_cat):
    g = load_golden("rqvae_c1")
    B, Din, D, H, K, L = (int(v) for v in g["shape"])
    x = I.randn(300, B, Din)
    if n_cat:
        x[:, -n_cat:] = (I.rand(301, B, n_cat) > 0.5).astype(np.float32)
    enc = I.mlp_weights(320, [Din, H, D])
    dec = I.mlp_weights(321, [D, H, Din])
    cbs = [(I.rand(330 + l, K, D) * (0.6 ** l) - (0.25 if l else 0.0)).astype(np.float32) for l in range(L)]
    if n_cat == 4:
        assert I.sha(*enc, *dec, *cbs) == str(g["sha"])
    us = [I.rand(310 + l, B, K) for l in range(L)]
    return g, x, enc, dec, cbs, us


@pytest.mark.parametrize("n_cat", [0, 4])
def test_rqvae_c1_eval(n_cat):
    g, x, enc, dec, cbs, _ = _c1(n_cat)
    res = O.mlp_forward(x, enc)
    so = O.rq_forward(res, cbs, O.STE, False, T, BETA)
    assert_ids_match(so.sem_ids, g[f"cat{n_cat}_eval_sem_ids"], res, cbs)
    same = (so.sem_ids == g[f"cat{n_cat}_eval_sem_ids"]).all(1)
    assert same.mean() > 0.995
    assert rel_err(so.embeddings[same], g[f"cat{n_cat}_eval_embeddings"][same]) < TOL
    assert np.abs(so.residuals[same] - g[f"cat{n_cat}_eval_residuals"][same]).max() < 1e-5
    assert rel_err(so.quantize_loss[same], g[f"cat{n_cat}_eval_qloss"][same]) < 1e-4
    if same.all():
        fo = O.rqvae_forward(x, enc, cbs, dec, O.STE, False, T, BETA, n_cat)
        ref = g[f"cat{n_cat}_eval_losses"]
        got = np.array([fo.loss, fo.reconstruction_loss, fo.rqvae_loss, fo.p_unique_ids])
        assert np.allclose(got, ref, rtol=TOL)
        assert rel_err(fo.embs_norm, g[f"cat{n_cat}_eval_embs_norm"]) < TOL


@pytest.mark.parametrize("n_cat", [0, 4])
@pytest.mark.parametrize("mname", ["ste", "rot", "gumbel"])
def test_rqvae_c1_train_losses(n_cat, mname):
    g, x, enc, dec, cbs, us = _c1(n_cat)
    fo = O.rqvae_forward(x, enc, cbs, dec, MODE[mname], True, T, BETA, n_cat, gumbel_uniform=us)
    ref = g[f"cat{n_cat}_{mname}_losses"]
    got = np.array([fo.loss, fo.reconstruction_loss, fo.rqvae_loss, fo.p_unique_ids])
    assert np.allclose(got, ref, rtol=1e-4), (got, ref)


@pytest.mark.parametrize("mname", ["eval", "ste", "rot"])
def test_rq_ns_chain(mname):
    g = load_golden("rq_ns2048")
    n, D, K, L = (int(v) for v in g["shape"])
    x, cbs = I.rq_problem(n, D, K, L, seed=1234)
    assert I.sha(x, *cbs) == str(g["sha"])
    so = O.rq_forward(x, cbs, MODE.get(mname, O.STE), mname != "eval", T, BETA)
    n_tie = assert_ids_match(so.sem_ids, g[f"{mname}_ids"], x, cbs)
    same = (so.sem_ids == g[f"{mname}_ids"]).all(1)
    assert n_tie <= 2
    assert rel_err(so.quantize_loss[same], g[f"{mname}_loss"][same]) < TOL
    assert rel_err(np.sqrt((so.embeddings ** 2).sum(1))[same], g[f"{mname}_embs_norm"][same]) < TOL
    assert np.abs(so.embeddings.sum(-1)[:32] - g[f"{mname}_embsum_head"])[same[:32]].max() < 1e-6
    ids = O.rq_tokenize(x, cbs)
    assert_ids_match(ids, g["eval_ids"], x, cbs)


def test_beauty_checkpoint_codebooks():
    g = load_golden("beauty_ckpt")
    cbs = list(g["codebooks"])
    so = O.rq_forward(g["res"], cbs, training=False, beta=BETA)
    n_tie = assert_ids_match(so.sem_ids, g["sem_ids"], g["res"], cbs)
    same = (so.sem_ids == g["sem_ids"]).all(1)
    assert n_tie <= 4
    assert rel_err(so.quantize_loss[same], g["qloss"][same]) < TOL
    assert rel_err(np.sqrt((so.embeddings ** 2).sum(1))[same], g["embs_norm"][same]) < TOL
    # a non-degenerate argmin workload (SURVEY 8c): most codes of every level are live
    assert all(len(np.unique(g["sem_ids"][:, l])) > 150 for l in range(3))


def test_mlp_and_l2norm():
    g = load_golden("mlp")
    ws = I.mlp_weights(500, [768, 512, 256, 128, 32])
    x = I.unit_rows(501, 256, 768)
    assert I.sha(x, *ws) == str(g["sha"])
    assert rel_err(O.mlp_forward(x, ws), g["y_norm0"]) < TOL
    assert rel_err(O.mlp_forward(x, ws, normalize=True), g["y_norm1"]) < TOL
    assert rel_err(O.l2norm(I.randn(503, 256, 40)), g["l2norm"]) < TOL


@pytest.mark.parametrize("tag,k,iters", [("a", 32, None), ("b", 256, 6), ("dup", 32, 4)])
def test_kmeans(tag, k, iters):
    g = load_golden("kmeans")
    x = {"a": lambda: I.randn(600, 4096, 16), "b": lambda: I.randn(601, 20000, 32),
         "dup": lambda: np.repeat(np.round(I.randn(602, 24, 8) * 8) / 8, 16, axis=0)}[tag]()
    assert I.sha(x) == str(g[f"{tag}_sha"])
    draws = list(g[f"{tag}_draws"])
    o = O.kmeans_run(x, k, g[f"{tag}_init_idx"], lambda n: draws.pop(0), max_iters=iters)
    assert len(draws) == 0
    agree = (o.assignment == g[f"{tag}_assignment"]).mean()
    assert agree > 0.999, agree
    assert np.abs(o.centroids - g[f"{tag}_centroids"]).max() < 2e-5


def test_gumbel():
    g = load_golden("gumbel")
    u, logits = I.rand(700, 64, 32), I.randn(701, 64, 32)
    assert rel_err(O.sample_gumbel_from_uniform(u), g["g"]) < TOL
    assert rel_err(O.gumbel_softmax_from_uniform(logits, 0.2, u), g["s"]) < 1e-4


def test_tokenizer_dedup_column():
    g = load_golden("tokenizer")
    N, Din, D, H, K, L = (int(v) for v in g["shape"])
    x = I.randn(801, N, Din)
    enc = I.mlp_weights(800, [Din, H, D])
    cbs = [(I.rand(810 + l, K, D) * (0.6 ** l) - (0.25 if l else 0.0)).astype(np.float32) for l in range(L)]
    assert I.sha(x, *enc, *cbs) == str(g["sha"])
    res = O.mlp_forward(x, enc)
    ids = O.rq_tokenize(res, cbs)
    ref = g["cached_ids"].astype(np.int64)
    assert_ids_match(ids, ref[:, :L], res, cbs)
    assert np.array_equal(O.dedup_rank(ref[:, :L]), ref[:, L])
    assert ref[:, L].max() > 3          # the fixture really exercises duplicates
    usage = O.codebook_usage(ref[:, :L], K)
    assert usage.sum(1).tolist() == [N] * L


def test_torch_cpu_port_matches_numpy_oracle_and_reference():
    """The torch-CPU port used for the CPU baseline timing gives the reference's ids."""
    import torch
    from oracle import rq_oracle_torch as OT
    g = load_golden("rq_ns2048")
    n, D, K, L = (int(v) for v in g["shape"])
    x, cbs = I.rq_problem(n, D, K, L, seed=1234)
    ids = OT.rq_tokenize(torch.from_numpy(x), [torch.from_numpy(c) for c in cbs]).numpy()
    assert_ids_match(ids, g["eval_ids"], x, cbs)
    assert_ids_match(ids, O.rq_tokenize(x, cbs), x, cbs)


def _beam_levels(g):
    B, k, H, K, N = (int(v) for v in g["shape"])
    nc = min(64, K)
    for h in range(H):
        logits = g[f"logits{h}"].astype(np.float64)
        e = np.exp(logits - logits.max(axis=1, keepdims=True))
        probas = (e / e.sum(axis=1, keepdims=True)).astype(np.float32)
        samples = g[f"prefix{h}"][:, -1].reshape(-1, nc)
        samp_log_p = np.log(np.take_along_axis(probas, samples, 1))
        yield h, samples, samp_log_p


def test_beam_oracle_vs_reference_generate():
    """oracle.check_valid_prefix / beam_select chained over the hierarchy levels reproduce the UNMODIFIED reference generate()
    (tests/golden/beam.npz: per-level validity masks, beams, cache-reorder indices, final beams and log-probabilities)."""
    g = load_golden("beam")
    B, k, H, K, N = (int(v) for v in g["shape"])
    corpus = g["corpus"]
    generated, log_probas = None, None
    for h, samples, samp_log_p in _beam_levels(g):
        assert np.array_equal(O.check_valid_prefix(corpus, g[f"prefix{h}"]), g[f"valid{h}"])
        if h > 0:
            assert np.array_equal(generated.reshape(-1, h), g[f"future{h}"])          # the beams the reference fed to its decoder
        generated, log_probas, parent = O.beam_select(corpus, samples, samp_log_p, generated, log_probas, k)
        if h > 0:
            assert np.array_equal(parent.reshape(-1), g[f"parent{h}"])
    assert np.array_equal(generated, g["generated"])
    np.testing.assert_allclose(log_probas, g["log_probas"], rtol=2e-5, atol=1e-6)
    for l in range(1, 5):
        assert np.array_equal(O.check_valid_prefix(g["v2_corpus"].astype(np.int64), g[f"v2_prefix{l}"]), g[f"v2_valid{l}"])
