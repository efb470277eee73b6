"""CPU tests of the host-side logic: drop-in aliasing of the reference's import paths, gin shim, tokenizer dedup,
sharding helpers, and the world_size-2 (gloo) paths of parallel.py with the kernel calls injected."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import inputs as I
from oracle import rq_oracle as O
from parity import load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_gin_shim_parses_the_reference_config_dialect():
    from rq_vae_recommender_b200 import gin_compat as gin
    from rq_vae_recommender_b200.modules.quantize import QuantizeForwardMode
    gin.clear_config()

    @gin.configurable
    def train(iterations=1, vae_hidden_dims=None, vae_codebook_mode=None, dataset_folder="", wandb_logging=True):
        return iterations, vae_hidden_dims, vae_codebook_mode, dataset_folder, wandb_logging

    gin.parse_config("""
import rq_vae_recommender_b200.modules.quantize
# a comment
train.iterations=400000
train.vae_hidden_dims=[512, 256, 128]
train.dataset_folder="dataset/amazon"
train.wandb_logging=False
train.vae_codebook_mode=%rq_vae_recommender_b200.modules.quantize.QuantizeForwardMode.STE
""")
    assert train() == (400000, [512, 256, 128], QuantizeForwardMode.STE, "dataset/amazon", False)
    assert train(iterations=3)[0] == 3
    gin.clear_config()


def test_dedup_rank_matches_oracle_and_reference_fixture():
    from rq_vae_recommender_b200.modules.tokenizer.semids import dedup_rank
    g = load_golden("tokenizer")
    ref = g["cached_ids"].astype(np.int64)
    L = ref.shape[1] - 1
    assert np.array_equal(dedup_rank(torch.from_numpy(ref[:, :L]), 8).numpy(), ref[:, L])
    ids = np.random.RandomState(0).randint(0, 3, size=(500, 3))
    assert np.array_equal(dedup_rank(torch.from_numpy(ids), 3).numpy(), O.dedup_rank(ids))
    assert dedup_rank(torch.zeros((0, 3), dtype=torch.int64), 256).shape == (0,)


def test_count_unique_matches_reference_expression():
    from rq_vae_recommender_b200.modules.rqvae import count_unique_id_tuples
    ids = torch.from_numpy(np.random.RandomState(1).randint(0, 4, size=(300, 3)))
    eq = (ids.unsqueeze(1) == ids.unsqueeze(0)).all(-1)                     # rqvae.py:159-167
    ref = (~torch.triu(eq, diagonal=1)).all(axis=1).sum().item()
    assert count_unique_id_tuples(ids, 4) == ref


def test_shard_bounds_cover_everything():
    from rq_vae_recommender_b200.parallel import shard_bounds
    for n in (0, 1, 7, 84000, 12101):
        for w in (1, 2, 3, 8):
            b = [shard_bounds(n, w, r) for r in range(w)]
            assert b[0][0] == 0 and b[-1][1] == n and all(b[i][1] == b[i + 1][0] for i in range(w - 1))
            assert max(h - l for l, h in b) - min(h - l for l, h in b) <= 1


def test_dropin_makes_the_unmodified_reference_import_the_replacements(tmp_path):
    """tests/golden/dropin.npz, read from the unmodified reference tree: its imports of the aliased modules
    (file:module:name), its RqVae / SemanticIdTokenizer calls (file:class:positional count:keywords), and the shipped
    Beauty checkpoint with its tensor payloads zeroed (pickle byte for byte)."""
    import inspect
    g = load_golden("dropin")
    root = tmp_path / "reference"                    # the reference's package skeleton: `modules` is a regular package
    (root / "modules").mkdir(parents=True)
    (root / "modules" / "__init__.py").write_text("")
    ckpt = tmp_path / "checkpoint_high_entropy.pt"
    ckpt.write_bytes(g["checkpoint"].tobytes())
    sys.modules.pop("gin", None)                     # let dropin register its own shim
    for k in [k for k in sys.modules if k.split(".")[0] in ("modules", "init", "distributions")]:
        del sys.modules[k]
    from rq_vae_recommender_b200 import dropin
    from rq_vae_recommender_b200.modules.tokenizer import semids as mine_semids
    import rq_vae_recommender_b200.modules.rqvae as mine
    try:
        aliased = dropin.install(reference_root=str(root))
        seen = set()
        for line in g["imports"]:
            path, module, name = str(line).split(":")
            if module not in aliased:                # imported from the reference tree untouched
                continue
            ns = {}
            exec(f"from {module} import {name}", ns)     # the reference's own import statement
            assert getattr(ns[name], "__module__", "").startswith("rq_vae_recommender_b200"), (path, module, name)
            seen.add((path, module, name))
        assert ("train_rqvae.py", "modules.rqvae", "RqVae") in seen
        assert ("modules/tokenizer/semids.py", "modules.rqvae", "RqVae") in seen
        # the reference's constructor calls bind to the replacement classes (the training script and its tokenizer)
        classes = {"RqVae": mine.RqVae, "SemanticIdTokenizer": mine_semids.SemanticIdTokenizer}
        for line in g["calls"]:
            path, cls, n_pos, kws = str(line).split(":")
            inspect.signature(classes[cls]).bind(*[None] * int(n_pos), **dict.fromkeys(kws.split(",")))
        assert any(str(line).startswith("modules/tokenizer/semids.py:RqVae:") for line in g["calls"])
        # a shipped checkpoint: state dict keys line up and the pickled model_config resolves to the replacements
        state = torch.load(str(ckpt), map_location="cpu", weights_only=False)
        m = mine.RqVae(input_dim=768, embed_dim=32, hidden_dims=[512, 256, 128], codebook_size=256,
                       codebook_kmeans_init=False, n_layers=3, n_cat_features=0)
        m.load_state_dict(state["model"])
        pickled_self = state["model_config"].get("self")
        assert pickled_self is None or type(pickled_self).__module__.startswith("rq_vae_recommender_b200")
    finally:
        dropin.uninstall()
        for k in [k for k in sys.modules if k.split(".")[0] in ("modules", "init", "distributions")]:
            del sys.modules[k]
        if str(root) in sys.path:
            sys.path.remove(str(root))


# ------------------------------------------------------------------ world_size = 2 over gloo, kernels injected (CPU)
def _cpu_make_buf(x, k):
    return dict(assign=torch.empty(x.shape[0], dtype=torch.int64), sums=torch.zeros((k, x.shape[1]), dtype=torch.float64),
                counts=torch.zeros(k, dtype=torch.int32), shift=torch.zeros(1))


def _cpu_assign_accumulate(x, c, buf):
    d = ((x[:, None, :] - c[None, :, :]) ** 2).sum(2)
    a = d.argmin(1)
    buf["assign"].copy_(a)
    buf["sums"].zero_().index_add_(0, a, x.double())
    buf["counts"].copy_(torch.bincount(a, minlength=c.shape[0]).int())


def _cpu_finalize(x, c, buf, reseed):
    nz = buf["counts"] > 0
    c[nz] = (buf["sums"][nz] / buf["counts"][nz].double().unsqueeze(1)).float()


def _worker(rank, world, port, n_total, k, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from rq_vae_recommender_b200 import parallel
    x = torch.from_numpy(I.randn(77, n_total, 8))
    lo, hi = parallel.shard_bounds(n_total, world, rank)
    np.random.seed(5); torch.manual_seed(6)
    cen, assign, iters = parallel.sharded_kmeans(x[lo:hi].clone(), k, n_total, max_iters=8,
                                                 assign_accumulate=_cpu_assign_accumulate, finalize=_cpu_finalize,
                                                 make_buf=_cpu_make_buf)
    ids_local = torch.stack([assign % 7, assign % 5], 1)
    full = parallel.all_gather_rows(ids_local.to(torch.int32), n_total).to(torch.int64)
    usage = parallel.codebook_usage(ids_local, 8, hist_fn=lambda ids, K: torch.stack(
        [torch.bincount(ids[:, l], minlength=K) for l in range(ids.shape[1])]))
    w = torch.zeros(k, 8)
    np.random.seed(5); torch.manual_seed(6)
    parallel.sharded_kmeans_init_(w, x[lo:hi].clone(), n_total, max_iters=8, assign_accumulate=_cpu_assign_accumulate,
                                  finalize=_cpu_finalize, make_buf=_cpu_make_buf)
    q.put((rank, cen.numpy(), full.numpy(), usage.numpy(), iters, w.numpy()))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_kmeans_and_gathers_world2_match_single_process():
    from rq_vae_recommender_b200 import parallel
    n_total, k = 1001, 16                      # odd: ragged shards
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, n_total, k, q)) for r in range(2)]
    [p.start() for p in procs]
    outs = sorted([q.get(timeout=120) for _ in procs], key=lambda t: t[0])
    [p.join(timeout=60) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    x = torch.from_numpy(I.randn(77, n_total, 8))
    np.random.seed(5); torch.manual_seed(6)
    cen1, assign1, iters1 = parallel.sharded_kmeans(x.clone(), k, n_total, max_iters=8,
                                                    assign_accumulate=_cpu_assign_accumulate, finalize=_cpu_finalize,
                                                    make_buf=_cpu_make_buf)
    for rank, cen, full, usage, iters, w in outs:
        assert iters == iters1
        assert np.allclose(cen, cen1.numpy(), atol=1e-6)           # every rank ends with the single-process centroids
        assert np.allclose(w, cen1.numpy(), atol=1e-6)
        ref_ids = torch.stack([assign1 % 7, assign1 % 5], 1).numpy()
        assert np.array_equal(full, ref_ids)                       # all-gathered id table is in corpus order
        assert np.array_equal(usage, O.codebook_usage(ref_ids, 8))
    assert np.array_equal(outs[0][1], outs[1][1])


def test_sharded_kmeans_windowed_host_checks_equal_per_iteration_checks():
    """The host is consulted once per window (check_every); a window that sees an empty cluster is rolled back and replayed with
    the reference's per-iteration RNG draws (init/kmeans.py:48-54), so both schedules give the same centroids.  Duplicated
    rows force duplicate initial centroids, i.e. empty clusters in the first iteration."""
    from rq_vae_recommender_b200 import parallel
    x = torch.from_numpy(I.randn(91, 64, 8))
    x = torch.cat([x, x[:32]], 0)              # 96 rows, a third of them duplicates
    outs = []
    for every in (1, 4):
        np.random.seed(11); torch.manual_seed(12)
        cen, assign, iters = parallel.sharded_kmeans(x.clone(), 48, x.shape[0], max_iters=12, check_every=every,
                                                     assign_accumulate=_cpu_assign_accumulate, finalize=_cpu_finalize,
                                                     make_buf=_cpu_make_buf)
        outs.append((cen.numpy(), assign.numpy().copy(), iters))
    assert np.allclose(outs[0][0], outs[1][0], atol=1e-6)
    assert np.array_equal(outs[0][1], outs[1][1])
    # no empties, converging data: the windowed loop may only run PAST convergence, never stop early
    y = torch.from_numpy(I.randn(92, 200, 8))
    res = []
    for every in (1, 4):
        np.random.seed(13); torch.manual_seed(14)
        cen, _, iters = parallel.sharded_kmeans(y.clone(), 8, 200, max_iters=40, check_every=every,
                                                assign_accumulate=_cpu_assign_accumulate, finalize=_cpu_finalize, make_buf=_cpu_make_buf)
        res.append((cen.numpy(), iters))
    assert res[0][1] == res[1][1] and np.allclose(res[0][0], res[1][0], atol=1e-6)


@pytest.mark.parametrize("mode_name,train", [("STE", True), ("ROTATION_TRICK", True), ("GUMBEL_SOFTMAX", True), ("STE", False)])
def test_forward_traces_to_one_graph_of_custom_operators(mode_name, train):
    """SURVEY 8(b): RqVae.forward (compiled by the reference, rqvae.py:141) exports as ONE graph (torch._dynamo.export raises on a
    graph break) whose kernel calls are rqb200:: custom operators.  Fake tensors only: no kernel runs, CPU is enough."""
    import torch
    import rq_vae_recommender_b200.library  # noqa: F401  (registers the operators)
    from rq_vae_recommender_b200.modules.rqvae import RqVae
    from rq_vae_recommender_b200.modules.quantize import QuantizeForwardMode as M
    from rq_vae_recommender_b200.data.schemas import SeqBatch
    m = RqVae(input_dim=64, embed_dim=16, hidden_dims=[32], codebook_size=32, codebook_kmeans_init=False,
              codebook_mode=getattr(M, mode_name), n_layers=2, commitment_weight=0.25, n_cat_features=4)
    m.train(train)

    def f(x):
        out = m(SeqBatch(None, None, None, x, None, None), 0.2)
        return out.loss, out.p_unique_ids, out.embs_norm

    gm = torch._dynamo.export(f)(torch.randn(48, 64)).graph_module
    names = {str(n.target) for n in gm.graph.nodes if n.op == "call_function" and "rqb200" in str(n.target)}
    level = "rqb200.gumbel_level_fwd.default" if (mode_name == "GUMBEL_SOFTMAX" and train) else "rqb200.rq_chain_fwd.default"
    assert names == {"rqb200.mlp_fwd.default", "rqb200.l2norm_fwd.default", "rqb200.count_unique_id_tuples.default", level}, names


def test_bench_reference_arm_contract(tmp_path):
    """`bench.py --impl reference` prints ONE JSON line with the keys of the GPU arm's line: the CPU port of the
    reference path on this host's cores, same metric / unit / workload string as the GPU arm, zero copy bytes.  With
    --dump-outputs it writes the last step's ids, which are the oracle's ids of the seeded batch."""
    import json
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--dump-outputs", str(tmp_path / "dump")], capture_output=True, text=True, timeout=600, cwd=root)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "rq_vae_items_per_sec" and d["unit"] == "items/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["n_gpus"] == 1
    assert "65536x768" in d["config"]["workload"] and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "items/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    import bench
    from parity import assert_ids_match
    ids = np.load(tmp_path / "dump" / "ids.npy")
    assert ids.dtype == np.float32 and ids.shape == (bench.N_ITEMS, bench.L)
    x, cbs = bench.make_problem(8192)                     # the codebooks are drawn from the first 8192 rows
    assert_ids_match(ids[:512].astype(np.int64), O.rq_tokenize(x[:512], cbs), x[:512], cbs)


@pytest.mark.parametrize("kw", [dict(codebook_sim_vq=True), dict(codebook_normalize=True),
                                dict(codebook_sim_vq=True, codebook_normalize=True)])
@pytest.mark.parametrize("mode_name", ["STE", "GUMBEL_SOFTMAX"])
def test_forward_traces_with_projected_and_normalised_codebooks(kw, mode_name):
    """The derived-codebook variants (sim_vq projection = an MLP op on the embedding table, row-normalised first level) also
    export as one graph."""
    import torch
    import rq_vae_recommender_b200.library  # noqa: F401
    from rq_vae_recommender_b200.modules.rqvae import RqVae
    from rq_vae_recommender_b200.modules.quantize import QuantizeForwardMode as M
    from rq_vae_recommender_b200.data.schemas import SeqBatch
    m = RqVae(input_dim=64, embed_dim=16, hidden_dims=[32], codebook_size=32, codebook_kmeans_init=False,
              codebook_mode=getattr(M, mode_name), n_layers=2, commitment_weight=0.25, n_cat_features=0, **kw)
    m.train()

    def f(x):
        out = m(SeqBatch(None, None, None, x, None, None), 0.2)
        return out.loss, out.p_unique_ids, out.embs_norm

    gm = torch._dynamo.export(f)(torch.randn(48, 64)).graph_module
    names = {str(n.target) for n in gm.graph.nodes if n.op == "call_function" and "rqb200" in str(n.target)}
    assert "rqb200.mlp_fwd.default" in names and "rqb200.count_unique_id_tuples.default" in names
    assert ("rqb200.gumbel_level_fwd.default" if mode_name == "GUMBEL_SOFTMAX" else "rqb200.rq_chain_fwd.default") in names
