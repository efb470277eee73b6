"""Generate tests/golden/*.npz by running the UNMODIFIED reference (from /root/reference) on seeded inputs.

Run in the build container only:   python tests/golden/make_golden.py
The GPU box never runs this (no /root/reference there); it consumes the committed .npz files.
The reference ships no tests or golden vectors (SURVEY 4), so these reference-generated outputs
are what pins the oracle (oracle/rq_oracle.py) and, through it, the CUDA path.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import inputs as I          # noqa: E402
import ref_harness          # noqa: E402

torch.set_num_threads(8)
ref = ref_harness.load()
Q = ref.quantize
MODES = {"ste": Q.QuantizeForwardMode.STE, "rot": Q.QuantizeForwardMode.ROTATION_TRICK,
         "gumbel": Q.QuantizeForwardMode.GUMBEL_SOFTMAX}
T = 0.2
BETA = 0.25


def t(a):
    return torch.from_numpy(np.ascontiguousarray(a))


def save(name, **arrs):
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **arrs)
    print(f"{name}: {os.path.getsize(path) / 1024:.0f} KB")


class InjectUniform:
    """Make distributions.gumbel.sample_gumbel consume an injected U (CPU mt19937 != CUDA Philox, SURVEY 4)."""
    def __init__(self, us):
        self.us = list(us)
    def __enter__(self):
        self.orig = ref.gumbel.torch.rand
        us = self.us
        def fake_rand(shape, device=None, **k):
            u = us.pop(0)
            assert tuple(u.shape) == tuple(shape)
            return u
        self.patch = fake_rand
        ref.gumbel.torch = _TorchProxy(torch, fake_rand)
        return self
    def __exit__(self, *a):
        ref.gumbel.torch = torch


class _TorchProxy:
    def __init__(self, mod, rand):
        self._m, self.rand = mod, rand
    def __getattr__(self, k):
        return getattr(self._m, k)


def make_quantize(D, K, cb, mode, beta=BETA):
    q = Q.Quantize(embed_dim=D, n_embed=K, do_kmeans_init=False, forward_mode=mode, commitment_weight=beta)
    with torch.no_grad():
        q.embedding.weight.copy_(t(cb))
    return q


# ------------------------------------------------------------------ G1: single-level Quantize, all modes, with grads
def g_quantize():
    """Full embeddings / input gradients are kept for the first `keep` rows only (the fixture stays under 1 MB); row sums
    cover every row."""
    out = {}
    for tag, (B, D, K, keep) in {"c1": (1024, 16, 32, 256), "d32": (1024, 32, 256, 128),
                                 "d768": (512, 768, 256, 16)}.items():
        x, cbs = I.rq_problem(B, D, K, 1, seed=100 + D)
        cb = cbs[0]
        g_out = I.randn(200 + D, B, D)
        g_loss = I.rand(201 + D, B)
        u = I.rand(202 + D, B, K)
        out[f"{tag}_shape"] = np.array([B, D, K, keep])
        out[f"{tag}_sha"] = np.array(I.sha(x, cb, g_out, g_loss, u))
        # eval
        q = make_quantize(D, K, cb, MODES["ste"]).eval()
        with torch.no_grad():
            o = q(t(x), temperature=T)
        out[f"{tag}_eval_ids"] = o.ids.numpy().astype(np.int16)
        out[f"{tag}_eval_loss"] = o.loss.numpy()
        out[f"{tag}_eval_emb"] = o.embeddings.numpy()[:keep]
        out[f"{tag}_eval_emb_rowsum"] = o.embeddings.double().sum(1).numpy()
        for mname, mode in MODES.items():
            q = make_quantize(D, K, cb, mode).train()
            xt = t(x).clone().requires_grad_(True)
            if mname == "gumbel":
                with InjectUniform([t(u)]):
                    o = q(xt, temperature=T)
            else:
                o = q(xt, temperature=T)
            ((o.embeddings * t(g_out)).sum() + (o.loss * t(g_loss)).sum()).backward()
            out[f"{tag}_{mname}_ids"] = o.ids.numpy().astype(np.int16)
            out[f"{tag}_{mname}_loss"] = o.loss.detach().numpy()
            out[f"{tag}_{mname}_emb"] = o.embeddings.detach().numpy()[:keep]
            out[f"{tag}_{mname}_emb_rowsum"] = o.embeddings.detach().double().sum(1).numpy()
            out[f"{tag}_{mname}_gx"] = xt.grad.numpy()[:keep]
            out[f"{tag}_{mname}_gx_rowsum"] = xt.grad.double().sum(1).numpy()
            gc = q.embedding.weight.grad.numpy()
            out[f"{tag}_{mname}_gc"] = gc if D <= 32 else gc[:, :32].copy()
            out[f"{tag}_{mname}_gc_rowsum"] = q.embedding.weight.grad.double().sum(1).numpy()
    save("quantize_levels", **out)


# ------------------------------------------------------------------ G2: RqVae C1 (BASELINE configs[0] shape)
def build_rqvae(Din, D, hidden, K, L, mode, n_cat, seed, normalize=False):
    m = ref.rqvae.RqVae(input_dim=Din, embed_dim=D, hidden_dims=list(hidden), codebook_size=K,
                        codebook_kmeans_init=False, codebook_normalize=normalize, codebook_mode=mode,
                        n_layers=L, commitment_weight=BETA, n_cat_features=n_cat)
    enc = I.mlp_weights(seed, [Din] + list(hidden) + [D])
    dec = I.mlp_weights(seed + 1, [D] + list(hidden)[::-1] + [Din])
    cbs = [I.rand(seed + 10 + l, K, D) * (0.6 ** l) - (0.25 if l else 0.0) for l in range(L)]
    cbs = [c.astype(np.float32) for c in cbs]
    with torch.no_grad():
        for lin, w in zip([mm for mm in m.encoder.mlp if isinstance(mm, torch.nn.Linear)], enc):
            lin.weight.copy_(t(w))
        for lin, w in zip([mm for mm in m.decoder.mlp if isinstance(mm, torch.nn.Linear)], dec):
            lin.weight.copy_(t(w))
        for layer, c in zip(m.layers, cbs):
            layer.embedding.weight.copy_(t(c))
    return m, enc, dec, cbs


def g_rqvae_c1():
    B, Din, D, hidden, K, L = 1024, 64, 16, [32], 32, 2
    out = {"shape": np.array([B, Din, D, hidden[0], K, L])}
    for n_cat in (0, 4):
        x = I.randn(300, B, Din)
        if n_cat:
            x[:, -n_cat:] = (I.rand(301, B, n_cat) > 0.5).astype(np.float32)
        batch = ref.schemas.SeqBatch(user_ids=None, ids=None, ids_fut=None, x=t(x), x_fut=None, seq_mask=None)
        us = [I.rand(310 + l, B, K) for l in range(L)]
        for mname, mode in MODES.items():
            m, enc, dec, cbs = build_rqvae(Din, D, hidden, K, L, mode, n_cat, seed=320)
            tag = f"cat{n_cat}_{mname}"
            if mname == "ste":
                m.eval()
                with torch.no_grad():
                    so = m.get_semantic_ids(t(x), T)
                    fo = m(batch, T)
                out[f"cat{n_cat}_eval_embeddings"] = so.embeddings.numpy()
                out[f"cat{n_cat}_eval_residuals"] = so.residuals.numpy()
                out[f"cat{n_cat}_eval_sem_ids"] = so.sem_ids.numpy().astype(np.int16)
                out[f"cat{n_cat}_eval_qloss"] = so.quantize_loss.numpy()
                out[f"cat{n_cat}_eval_losses"] = np.array([fo.loss.item(), fo.reconstruction_loss.item(),
                                                           fo.rqvae_loss.item(), fo.p_unique_ids.item()])
                out[f"cat{n_cat}_eval_embs_norm"] = fo.embs_norm.numpy()
            m.train()
            if mname == "gumbel":
                with InjectUniform([t(u) for u in us]):
                    fo = m(batch, T)
            else:
                fo = m(batch, T)
            fo.loss.backward()
            out[f"{tag}_losses"] = np.array([fo.loss.item(), fo.reconstruction_loss.item(),
                                             fo.rqvae_loss.item(), fo.p_unique_ids.item()])
            out[f"{tag}_embs_norm"] = fo.embs_norm.detach().numpy()
            for name, p in m.named_parameters():
                out[f"{tag}_grad_{name}"] = p.grad.numpy()
    out["sha"] = np.array(I.sha(*enc, *dec, *cbs))
    save("rqvae_c1", **out)


# ------------------------------------------------------------------ G3: north-star shaped chain, quantizer fed D=768 directly
def g_rq_ns():
    n, D, K, L = 2048, 768, 256, 3
    x, cbs = I.rq_problem(n, D, K, L, seed=1234)
    out = {"shape": np.array([n, D, K, L]), "sha": np.array(I.sha(x, *cbs))}
    for mname in ("eval", "ste", "rot"):
        mode = MODES.get(mname, MODES["ste"])
        layers = [make_quantize(D, K, cb, mode) for cb in cbs]
        res = t(x)
        ids, embs, loss = [], [], 0
        with torch.no_grad():
            for q in layers:
                q.train(mname != "eval")
                o = q(res, temperature=T)
                loss = loss + o.loss
                res = res - o.embeddings
                ids.append(o.ids)
                embs.append(o.embeddings)
        e = torch.stack(embs, -1)
        out[f"{mname}_ids"] = torch.stack(ids, -1).numpy().astype(np.int16)
        out[f"{mname}_loss"] = loss.numpy()
        out[f"{mname}_embs_norm"] = e.norm(dim=1).numpy()
        out[f"{mname}_embsum_head"] = e.sum(-1).numpy()[:32]
        out[f"{mname}_final_res_rowsum"] = res.double().sum(1).numpy()
    save("rq_ns2048", **out)


# ------------------------------------------------------------------ G4: real weights (shipped Beauty checkpoint), D=32
def g_beauty():
    path = os.path.join(ref_harness.REFERENCE, "trained_models/rqvae_amazon_beauty/checkpoint_high_entropy.pt")
    state = torch.load(path, map_location="cpu", weights_only=False)
    sd = state["model"]
    m = ref.rqvae.RqVae(input_dim=768, embed_dim=32, hidden_dims=[512, 256, 128], codebook_size=256,
                        codebook_kmeans_init=False, codebook_mode=MODES["rot"], n_layers=3, n_cat_features=0)
    m.load_state_dict(sd)
    m.eval()
    n = 4096
    x = I.unit_rows(77, n, 768)
    with torch.no_grad():
        res = m.encode(t(x))
        so = m.get_semantic_ids(t(x), T)
    cbs = np.stack([sd[f"layers.{i}.embedding.weight"].numpy() for i in range(3)])
    save("beauty_ckpt", codebooks=cbs, res=res.numpy(), sem_ids=so.sem_ids.numpy().astype(np.int16),
         qloss=so.quantize_loss.numpy(), embs_norm=so.embeddings.norm(dim=1).numpy(),
         iter=np.array(state["iter"]))


# ------------------------------------------------------------------ G5: MLP + l2norm
def g_mlp():
    """gx is kept for the first 32 of the 256 rows (the fixture stays under 1 MB); its row sums cover every row."""
    dims = [768, 512, 256, 128, 32]
    ws = I.mlp_weights(500, dims)
    x = I.unit_rows(501, 256, 768)
    out = {"sha": np.array(I.sha(x, *ws))}
    for norm in (False, True):
        mlp = ref.encoder.MLP(input_dim=768, hidden_dims=dims[1:-1], out_dim=32, normalize=norm)
        with torch.no_grad():
            for lin, w in zip([mm for mm in mlp.mlp if isinstance(mm, torch.nn.Linear)], ws):
                lin.weight.copy_(t(w))
        xt = t(x).clone().requires_grad_(True)
        y = mlp(xt)
        gy = I.randn(502, 256, 32)
        (y * t(gy)).sum().backward()
        out[f"y_norm{int(norm)}"] = y.detach().numpy()
        out[f"gx_norm{int(norm)}"] = xt.grad.numpy()[:32]
        out[f"gx_rowsum_norm{int(norm)}"] = xt.grad.double().sum(1).numpy()
        out[f"gw3_norm{int(norm)}"] = mlp.mlp[6].weight.grad.numpy()
        out[f"gw0_rowsum_norm{int(norm)}"] = mlp.mlp[0].weight.grad.double().sum(1).numpy()
    out["l2norm"] = ref.normalize.l2norm(t(x[:, :40] * 0.0 + I.randn(503, 256, 40))).numpy()
    save("mlp", **out)


# ------------------------------------------------------------------ G6: k-means init
def g_kmeans():
    out = {}
    draws = []
    orig_randint = torch.randint
    def rec_randint(*a, **k):
        r = orig_randint(*a, **k)
        draws.append(int(r))
        return r
    for tag, x, k, iters in (("a", I.randn(600, 4096, 16), 32, None),
                             ("b", I.randn(601, 20000, 32), 256, 6),
                             ("dup", np.repeat(np.round(I.randn(602, 24, 8) * 8) / 8, 16, axis=0), 32, 4)):
        np.random.seed(610)
        torch.manual_seed(611)
        st = np.random.get_state()
        init_idx = np.random.choice(x.shape[0], k, replace=False)
        np.random.set_state(st)
        draws.clear()
        ref.kmeans.torch = _KmTorchProxy(torch, rec_randint)
        km = ref.kmeans.Kmeans(k=k, max_iters=iters)
        o = km.run(t(x))
        ref.kmeans.torch = torch
        out[f"{tag}_init_idx"] = init_idx
        out[f"{tag}_centroids"] = o.centroids.numpy()
        out[f"{tag}_assignment"] = o.assignment.numpy().astype(np.int16)
        out[f"{tag}_draws"] = np.array(draws, np.int64)
        out[f"{tag}_sha"] = np.array(I.sha(x))
        print("kmeans", tag, "draws", len(draws))
    # kmeans_init_ writes in place
    w = torch.zeros(32, 16)
    np.random.seed(610)
    ref.kmeans.kmeans_init_(w, t(I.randn(600, 4096, 16)))
    assert np.array_equal(w.numpy(), out["a_centroids"])
    save("kmeans", **out)


class _KmTorchProxy:
    def __init__(self, mod, randint):
        self._m, self.randint = mod, randint
    def __getattr__(self, k):
        return getattr(self._m, k)


# ------------------------------------------------------------------ G7: gumbel
def g_gumbel():
    u = I.rand(700, 64, 32)
    logits = I.randn(701, 64, 32)
    with InjectUniform([t(u), t(u)]):
        g = ref.gumbel.sample_gumbel(u.shape, device="cpu")
        s = ref.gumbel.gumbel_softmax_sample(t(logits), 0.2, device="cpu")
    ts = ref.gumbel.TemperatureScheduler(t0=1.0, min_t=0.1, anneal_rate=0.001, step_size=10)
    temps = np.array([ts.get_t(i) for i in range(100)])
    save("gumbel", g=g.numpy(), s=s.numpy(), temps=temps)


# ------------------------------------------------------------------ G8: tokenizer corpus pass (dedup column)
def g_tokenizer():
    N, Din, D, hidden, K, L = 1500, 64, 16, [32], 8, 2
    m, enc, dec, cbs = build_rqvae(Din, D, hidden, K, L, MODES["gumbel"], 0, seed=800)
    x = I.randn(801, N, Din)
    tok = ref.semids.SemanticIdTokenizer(input_dim=Din, output_dim=D, hidden_dims=hidden, codebook_size=K,
                                         n_layers=L, n_cat_feats=0)
    tok.rq_vae = m

    class FakeItems:
        def __len__(self):
            return N
        def __getitem__(self, idx):
            idx = torch.as_tensor(idx)
            return ref.schemas.SeqBatch(user_ids=-1 * torch.ones_like(idx), ids=idx.unsqueeze(0),
                                        ids_fut=-1 * torch.ones_like(idx), x=t(x)[idx],
                                        x_fut=-1 * torch.ones_like(idx), seq_mask=torch.ones_like(idx, dtype=bool))
    cached = tok.precompute_corpus_ids(FakeItems())
    save("tokenizer", cached_ids=cached.numpy().astype(np.int16), sha=np.array(I.sha(x, *enc, *cbs)),
         shape=np.array([N, Din, D, hidden[0], K, L]))


def g_beam():
    """Constrained beam search, data side (modules/model.py:169-182, :300-391).  The UNMODIFIED `generate` and
    `_check_valid_prefix` of EncoderDecoderRetrievalModel run on a stand-in `self`: the transformer passes return seeded random
    activations (the decoder step itself is not part of this fixture), everything the search does with them -- sampling, prefix
    validity against the corpus, scoring, sort, top-k, parent gather, cache reorder index -- is the reference's code.  Recorded
    per hierarchy level: the logits, the sampled tokens, the validity mask, the beams entering the level, the reorder index;
    and the final beams and log-probabilities."""
    import importlib
    import types as _types
    stub = sys.modules.pop("accelerate", None)              # transformers probes the real package: the harness stub has no spec
    try:
        M = importlib.import_module("modules.model")
    finally:
        if stub is not None:
            sys.modules["accelerate"] = stub
    B, k, H, K, N, d = 6, 5, 4, 16, 300, 8
    rs = np.random.RandomState(900)
    corpus = rs.randint(0, K, size=(N, H)).astype(np.int64)
    corpus[:, 0] = rs.randint(0, 6, size=N)                   # a few first-level ids never occur: invalid candidates exist
    rec = dict(logits=[], prefix=[], valid=[], future=[], parent=[])

    class FakeCache:
        def __init__(self, *a, **kw):
            pass
        def reorder_cache(self, idx):
            rec["parent"].append(idx.clone())
    class Head(torch.nn.Module):
        def __init__(self, seed):
            super().__init__()
            g = torch.Generator().manual_seed(seed)
            self.w = torch.randn(d, K, generator=g) * 1.5
        def forward(self, x):
            out = x @ self.w
            rec["logits"].append(out.clone())
            return out
    fake = _types.SimpleNamespace(top_k_for_generation=k, num_embeddings_per_hierarchy=K, num_hierarchies=H,
                                  codebooks=t(corpus), decoder_mlp=[Head(910 + h) for h in range(H)])
    gen = torch.Generator().manual_seed(901)
    def encoder_forward_pass(attention_mask, input_ids, user_id=None):
        return torch.randn(B, 3, d, generator=gen), torch.ones(B, 3, dtype=torch.bool)
    def decoder_forward_pass(future_ids, encoder_output, attention_mask_for_encoder, use_cache, past_key_values):
        rows = encoder_output.shape[0]
        rec["future"].append(None if future_ids is None else future_ids.clone())
        return torch.randn(rows, 1, d, generator=gen), past_key_values
    def check(prefix, batch_size=100000):
        out = M.EncoderDecoderRetrievalModel._check_valid_prefix(fake, prefix, batch_size)
        rec["prefix"].append(prefix.clone()); rec["valid"].append(out.clone())
        return out
    fake.encoder_forward_pass, fake.decoder_forward_pass, fake._check_valid_prefix = encoder_forward_pass, decoder_forward_pass, check
    orig = (M.EncoderDecoderCache, M.DynamicCache)
    M.EncoderDecoderCache, M.DynamicCache = FakeCache, FakeCache
    try:
        torch.manual_seed(902)                                # torch.multinomial inside generate
        generated, log_probas = M.EncoderDecoderRetrievalModel.generate.__wrapped__(fake, None, torch.zeros(B, 1, dtype=torch.long)) \
            if hasattr(M.EncoderDecoderRetrievalModel.generate, "__wrapped__") else \
            M.EncoderDecoderRetrievalModel.generate(fake, None, torch.zeros(B, 1, dtype=torch.long))
    finally:
        M.EncoderDecoderCache, M.DynamicCache = orig
    out = dict(corpus=corpus, shape=np.array([B, k, H, K, N]), generated=generated.numpy(), log_probas=log_probas.numpy())
    for h in range(H):
        out[f"logits{h}"] = rec["logits"][h].numpy()
        out[f"prefix{h}"] = rec["prefix"][h].numpy()
        out[f"valid{h}"] = rec["valid"][h].numpy()
        if h > 0:
            out[f"future{h}"] = rec["future"][h].numpy()
            out[f"parent{h}"] = rec["parent"][h - 1].numpy()
    # a larger validity-only case: every prefix length, present and absent prefixes, ids outside [0, K)
    corpus2 = rs.randint(0, 256, size=(5000, 4)).astype(np.int64)
    corpus2[:, 3] = rs.randint(0, 3, size=5000)
    fake2 = _types.SimpleNamespace(codebooks=t(corpus2))
    for l in range(1, 5):
        pres = corpus2[rs.randint(0, 5000, size=400), :l]
        absent = rs.randint(0, 256, size=(400, l)).astype(np.int64)
        odd = pres.copy()[:20]; odd[:, -1] = np.array([-1, 256, 300, 1 << 40] * 5)
        pf = np.concatenate([pres, absent, odd])
        out[f"v2_prefix{l}"] = pf
        out[f"v2_valid{l}"] = M.EncoderDecoderRetrievalModel._check_valid_prefix(fake2, t(pf)).numpy()
    out["v2_corpus"] = corpus2.astype(np.int16)
    save("beam", **out)


# ------------------------------------------------------------------ G9: what dropin.py must satisfy
def g_dropin():
    """Read from the unmodified tree: every `from modules.* / init.* / distributions.* import name` (file:module:name), the
    RqVae / SemanticIdTokenizer calls (file:class:positional count:keywords), and the shipped Beauty checkpoint with its
    tensor payloads zeroed -- the pickle (class paths, model_config, state-dict layout) is kept byte for byte, and the zeros
    compress to a few KB."""
    import ast
    import io
    import zipfile
    root = ref_harness.REFERENCE
    imports, calls = [], []
    for dirpath, dirs, files in os.walk(root):
        dirs.sort()
        for f in sorted(files):
            if not f.endswith(".py"):
                continue
            rel = os.path.relpath(os.path.join(dirpath, f), root)
            with open(os.path.join(dirpath, f)) as fh:
                tree = ast.parse(fh.read())
            for node in ast.walk(tree):
                if isinstance(node, ast.ImportFrom) and node.module and node.module.split(".")[0] in (
                        "modules", "init", "distributions"):
                    imports += [f"{rel}:{node.module}:{a.name}" for a in node.names]
                elif isinstance(node, ast.Call) and getattr(node.func, "id", None) in ("RqVae", "SemanticIdTokenizer"):
                    calls.append(f"{rel}:{node.func.id}:{len(node.args)}:" + ",".join(k.arg for k in node.keywords if k.arg))
    buf = io.BytesIO()
    path = os.path.join(root, "trained_models/rqvae_amazon_beauty/checkpoint_high_entropy.pt")
    with zipfile.ZipFile(path) as src, zipfile.ZipFile(buf, "w", zipfile.ZIP_STORED) as dst:
        for info in src.infolist():
            data = src.read(info.filename)
            if "/data/" in info.filename:                     # <archive>/data/<key>: one tensor storage each
                data = bytes(len(data))
            dst.writestr(info.filename, data)
    save("dropin", imports=np.array(imports), calls=np.array(calls), checkpoint=np.frombuffer(buf.getvalue(), np.uint8))


if __name__ == "__main__":
    which = sys.argv[1:] or ["quantize", "rqvae_c1", "rq_ns", "beauty", "mlp", "kmeans", "gumbel", "tokenizer", "beam",
                             "dropin"]
    for w in which:
        globals()["g_" + w]()
