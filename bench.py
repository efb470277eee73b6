#!/usr/bin/env python
"""bench.py -- BASELINE.json metric: RQ-VAE items/sec for the fused L-level quantiser (64K x 768, K=256, L=3).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (tokenise: L chained distance+argmin levels) over one batch of 65 536
synthetic unit-norm item vectors per GPU.  Prints ONE JSON line (rank 0).  Under torchrun every rank tokenises its
own shard (items are independent: weak scaling, no data-path collective); the time is the max over ranks.

  value     items/s with the batch already resident in HBM (CUDA events around the K steps)
  e2e       items/s through the public host API (pinned host rows -> H2D -> kernels -> D2H ids inside the timing)
  roofline  algorithmic HBM bytes of the dominant kernel / its event-timed duration vs MEASURED_PEAKS.json
  cpu_baseline  the torch-CPU port of the reference path (oracle/rq_oracle_torch.py) on this host's cores, bounded sample
  prepare_ms    one-time cost of the frozen-codebook state (fp16 images, float64 Gram tables), outside the timed steps
  c3            (N > 1) BASELINE config 3: an 84 000-item corpus sharded over the ranks: local tokenise + all-gather of the
                int32 id blocks + all-reduce of the [L,K] usage counts per step (eager, and replayed as ONE CUDA graph), checked against one GPU tokenising the whole
                corpus; plus one Lloyd iteration (assign + fp64 accumulate + all-reduce + update) at 20 000 x 32 and x 768

  c2            (N = 1) BASELINE config 2: 12 101 x 768 items, device-timed through the module-API routing (ops.rq_tokenize_auto)
  pipeline      (N = 1) the shipped architecture: 768-512-256-128-32 encoder (split-precision tensor-core GEMMs) + 3-level RQ at
                D = 32, 65 536 items, index-exact precision: encoder ms, tokenise ms, id agreement with the CUDA-core SGEMM path

  c4            (N = 1) BASELINE config 4 shapes, fp32 I/O: a 3-level Gumbel-softmax chain and the rotation-trick chain at
                65 536 x 768, forward and forward + backward, device-timed, with the train-forward algorithmic bytes of SURVEY 8(d)

--impl reference times that CPU port as the reference arm (the reference is pure Python/PyTorch: there is nothing
to compile into oracle/_ref, see DESIGN.md).

--dump-outputs DIR writes what the last timed step returned -- the [65 536, L] semantic ids -- as DIR/ids.npy (float32,
exact for ids < 2^24; DIR/ids_rank<r>.npy per rank under torchrun).  The inputs are seeded, so two builds (or the two
--impl arms) run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))

N_ITEMS, D, K, L = 65536, 768, 256, 3
METRIC = "rq_vae_items_per_sec"
UNIT = "items/s"
WORKLOAD = f"rq_tokenize {N_ITEMS}x{D} fp32, K={K}, L={L} (north-star shape of BASELINE.json metric)"


def make_problem(n_items, seed=1234):
    import inputs as I
    x = I.unit_rows(seed, n_items, D)
    _, cbs = I.rq_problem(8192, D, K, L, seed=seed, x=x[:8192])
    return x, cbs


def dump_outputs(out_dir, arrays):
    """arrays: name -> tensor or array; each is written as out_dir/<name>.npy in float32."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


def algorithmic_bytes(n_items):
    """SURVEY 8(d): 4*D read + 8*L written per item, + the L*K*D fp32 codebooks once per launch."""
    return n_items * (4 * D + 8 * L) + 4 * L * K * D


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except (ValueError, IndexError):
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


_BEST_THREADS = None


def cpu_threads(x=None, cbt=None):
    """Thread count at which the reference's CPU path runs FASTEST on this host.  More threads is not always faster for
    these memory-bound ops (128 threads measured 3x slower than 8-32 on the B200 host), and the fair baseline is the
    reference at its best, so a few counts are timed on a full-size pass and the best is kept."""
    global _BEST_THREADS
    import torch
    if _BEST_THREADS is not None or x is None:
        torch.set_num_threads(_BEST_THREADS or (os.cpu_count() or 1))
        return torch.get_num_threads()
    from oracle import rq_oracle_torch as OT
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (4, 8, 16, 32, 64, ncpu) if c <= ncpu})
    best, best_t = cands[0], float("inf")
    for c in cands:          # min of 3: single samples are dominated by page-fault noise (observed 8K..100K items/s)
        torch.set_num_threads(c)
        OT.rq_tokenize(x[:16384], cbt)
        dt = float("inf")
        for _ in range(3):
            t0 = time.perf_counter()
            OT.rq_tokenize(x[:16384], cbt)
            dt = min(dt, time.perf_counter() - t0)
        if dt < best_t:
            best, best_t = c, dt
    _BEST_THREADS = best
    torch.set_num_threads(best)
    return best


def cpu_port_items_per_sec(x, cbs, budget_s=12.0, sample=65536):
    """The reference's CPU path (torch-CPU port, op for op quantize.py:113-128 + rqvae.py:125-132, eager fp32, all host
    threads) on a bounded sample of the same workload."""
    import torch
    from oracle import rq_oracle_torch as OT
    xs = torch.from_numpy(x[:sample])
    cbt = [torch.from_numpy(c) for c in cbs]
    threads = cpu_threads(xs, cbt)
    OT.rq_tokenize(xs, cbt)                   # full-size warm-up: steady state, not first-touch page faults
    t0 = time.perf_counter()
    n, best = 0, float("inf")
    while True:
        t1 = time.perf_counter()
        OT.rq_tokenize(xs, cbt)
        best = min(best, time.perf_counter() - t1)
        n += len(xs)
        dt = time.perf_counter() - t0
        if dt > budget_s or n >= 16 * sample:
            break
    return (n / dt, threads, f"{n} items ({n // len(xs)} passes over {len(xs)} rows of the same synthetic batch), {dt:.1f}s; "
            f"fastest pass {len(xs) / best:.0f} items/s (host timing is noisy: ~470 MB of temporaries are re-faulted per pass)")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from oracle import rq_oracle_torch as OT
    sample = 65536
    x, cbs = make_problem(sample)
    xt, cbt = torch.from_numpy(x), [torch.from_numpy(c) for c in cbs]
    cores = cpu_threads(xt, cbt)
    for _ in range(max(args.warmup, 1)):      # full-size warm-up: steady state, not first-touch page faults
        OT.rq_tokenize(xt, cbt)
    t0 = time.perf_counter()
    best = float("inf")
    ids = None
    for _ in range(args.steps):
        t1 = time.perf_counter()
        ids = OT.rq_tokenize(xt, cbt)
        best = min(best, time.perf_counter() - t1)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"ids": ids})
    val = args.steps * sample / dt
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": f"{sample} rows per step",
                   "best_step_items_per_sec": sample / best},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{args.steps} steps x {sample} rows of the same synthetic batch (torch CPU eager fp32, best of several thread counts)"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def run_c3(world, rank, cbs, torch, dist, ops, parallel):
    """BASELINE.json config 3: ~84K items x 768 tokenised across the ranks with the collectives north_star names
    (modules/tokenizer/semids.py:76-110 corpus pass, train_rqvae.py:285-289 usage counts, init/kmeans.py:39-70 Lloyd update)."""
    import inputs as I
    n3 = 84000
    x_all = I.unit_rows(4321, n3, D)                       # same corpus on every rank (seeded), each keeps its shard
    lo, hi = parallel.shard_bounds(n3, world, rank)
    xs = torch.from_numpy(x_all[lo:hi]).cuda()
    tok = parallel.CorpusTokenizer(cbs)

    def step():
        ids_local = tok.tokenize_device(xs)
        table = parallel.all_gather_rows(ids_local.to(torch.int32), n3)
        usage = parallel.codebook_usage(ids_local, K)
        return table, usage

    for _ in range(5):
        table, usage = step()
    torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
    steps = 200
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        table, usage = step()
    e1.record()
    torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
    ms_rank = torch.tensor([e0.elapsed_time(e1) / steps], device="cuda")
    per_rank = [torch.zeros_like(ms_rank) for _ in range(world)]
    dist.all_gather(per_rank, ms_rank)
    per_rank = [float(t.item()) for t in per_rank]
    # one GPU tokenising the whole corpus: the strong-scaling reference AND the parity check of the sharded table
    out = {"items": n3, "steps": steps, "ms_per_step_per_rank": per_rank, "ms_per_step": max(per_rank),
           "items_per_sec": n3 / (max(per_rank) * 1e-3),
           "timed": "local tokenise + all_gather(int32 ids) + all_reduce([L,K] usage), eager launches, NCCL"}
    # the same step captured in ONE CUDA graph (kernel + both collectives): what a serving loop would replay.  Every rank must
    # agree that its capture succeeded before anybody replays (a captured collective replayed by one rank only would hang).
    ok_flag = torch.ones(1, device="cuda")
    graph = None
    try:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            table_g, usage_g = step()
    except Exception as e:                                   # capture not possible here: keep the eager record
        ok_flag[0] = 0.0
        out["graph_error"] = f"{type(e).__name__}: {e}"[:200]
        graph = None
    torch.cuda.synchronize()
    dist.all_reduce(ok_flag, op=dist.ReduceOp.MIN)
    if bool(ok_flag.item() == 1.0):
        for _ in range(5):
            graph.replay()
        torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
        e0.record()
        for _ in range(steps):
            graph.replay()
        e1.record()
        torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
        g_ms = torch.tensor([e0.elapsed_time(e1) / steps], device="cuda")
        per_g = [torch.zeros_like(g_ms) for _ in range(world)]
        dist.all_gather(per_g, g_ms)
        out["graph_ms_per_step_per_rank"] = [float(t.item()) for t in per_g]
        out["graph_ms_per_step"] = max(out["graph_ms_per_step_per_rank"])
        out["graph_tables_equal_eager"] = bool(torch.equal(table_g, table)) and bool(torch.equal(usage_g, usage))
    match = torch.zeros(1, device="cuda")
    if rank == 0:
        xf = torch.from_numpy(x_all).cuda()
        for _ in range(5):
            full = tok.tokenize_device(xf)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(50):
            full = tok.tokenize_device(xf)
        e1.record()
        torch.cuda.synchronize()
        out["single_gpu_ms"] = e0.elapsed_time(e1) / 50
        out["speedup_vs_single_gpu"] = out["single_gpu_ms"] / out["ms_per_step"]
        if "graph_ms_per_step" in out:
            out["graph_speedup_vs_single_gpu"] = out["single_gpu_ms"] / out["graph_ms_per_step"]
        ok = bool(torch.equal(full.to(torch.int32), table)) and bool(torch.equal(ops.sid_histogram(full, K), usage))
        match[0] = 1.0 if ok else 0.0
        del xf
    dist.broadcast(match, src=0)
    out["sharded_ids_match_single"] = bool(match.item() == 1.0)
    # one Lloyd iteration with its all-reduce (init/kmeans.py:39-58), shapes of train_rqvae.py:179-181
    out["kmeans_lloyd_iteration_ms"] = {}
    for dk in (32, D):
        n_k = 20000
        xk_all = I.unit_rows(99, n_k, dk)
        klo, khi = parallel.shard_bounds(n_k, world, rank)
        xk = torch.from_numpy(xk_all[klo:khi]).cuda()
        cen = torch.from_numpy(xk_all[:K].copy()).cuda()
        buf = ops.kmeans_workspace(xk, K)

        def lloyd():
            ops.kmeans_assign_accumulate(xk, cen, buf)
            dist.all_reduce(buf["sums"]); dist.all_reduce(buf["counts"])
            ops.kmeans_finalize(xk, cen, buf, None)

        for _ in range(5):
            lloyd()
        torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
        e0.record()
        for _ in range(50):
            lloyd()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / 50], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out["kmeans_lloyd_iteration_ms"][f"20000x{dk}"] = float(t.item())
    return out


def _event_ms(torch, fn, n=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def run_c2(x, cbs, torch, ops):
    """BASELINE configs[1]: ~12K x 768 items on one B200, through the routing the module API uses."""
    n = 12101
    xs = x[:n].contiguous()
    with torch.no_grad():
        ms = _event_ms(torch, lambda: ops.rq_tokenize_auto(xs, cbs), n=20)
        same = bool(torch.equal(ops.rq_tokenize_auto(xs, cbs), ops.rq_tokenize(xs, cbs)))
    return {"items": n, "ms": ms, "items_per_sec": n / (ms * 1e-3), "ids_equal_exact_kernel": same,
            "timed": "ops.rq_tokenize_auto (cached prepared state), device resident"}


def run_pipeline(torch, ops):
    """Shipped architecture end to end on the device: encoder MLP 768-512-256-128-32 + 3-level RQ (K = 256, D = 32), 65 536 items,
    default (index-exact) precision.  Codebooks are k-means-initialised on the encoder outputs of clustered synthetic items, so
    the codes are live and id agreement is meaningful."""
    from rq_vae_recommender_b200.modules.rqvae import RqVae
    from rq_vae_recommender_b200.modules.quantize import QuantizeForwardMode
    from rq_vae_recommender_b200.data.schemas import SeqBatch
    torch.manual_seed(0)
    np.random.seed(0)
    m = RqVae(input_dim=768, embed_dim=32, hidden_dims=[512, 256, 128], codebook_size=256, codebook_kmeans_init=True,
              codebook_mode=QuantizeForwardMode.STE, n_layers=3, n_cat_features=0).cuda()
    g = torch.Generator(device="cuda").manual_seed(1)
    centers = torch.nn.functional.normalize(torch.randn(200, 768, device="cuda", generator=g), dim=1)

    def items(n):
        v = centers[torch.randint(0, 200, (n,), device="cuda", generator=g)]
        v = v + 0.5 * torch.nn.functional.normalize(torch.randn(n, 768, device="cuda", generator=g), dim=1)
        return torch.nn.functional.normalize(v, dim=1)

    m.train()
    with torch.no_grad():
        m(SeqBatch(None, None, None, items(20000), None, None), 0.2)     # lazy k-means init (train_rqvae.py:178-183)
    m.eval()
    x = items(N_ITEMS)
    with torch.no_grad():
        enc_ms = _event_ms(torch, lambda: m.encode(x))
        tok_ms = _event_ms(torch, lambda: m.tokenize(x))
        ids = m.tokenize(x)
        calls0 = ops.SPLIT_CALLS
        m.encode(x)
        on_tc = ops.SPLIT_CALLS - calls0
        old, ops.SPLIT_MIN_ROWS = ops.SPLIT_MIN_ROWS, 1 << 62            # the CUDA-core SGEMM path for comparison
        try:
            sg_ms = _event_ms(torch, lambda: m.encode(x), n=2, warm=1)
            ids_sg = m.tokenize(x)
        finally:
            ops.SPLIT_MIN_ROWS = old
    flop = 2.0 * N_ITEMS * (768 * 512 + 512 * 256 + 256 * 128 + 128 * 32)
    return {"items": N_ITEMS, "encoder_ms": enc_ms, "tokenize_ms": tok_ms, "items_per_sec": N_ITEMS / (tok_ms * 1e-3),
            "encoder_tflops_fp32_equivalent": flop / (enc_ms * 1e-3) / 1e12, "encoder_gemms_on_tensor_cores": on_tc,
            "encoder_ms_cuda_core_sgemm": sg_ms,
            "ids_rows_equal_sgemm_path": float((ids == ids_sg).all(1).float().mean().item()),
            "unique_id_tuples": int(torch.unique(ids, dim=0).shape[0])}


def run_c4(x, cbs, torch, ops):
    """BASELINE configs[3]: the training-mode paths at 64K x 768 (fp32 I/O; a bf16-I/O variant is not built).  Algorithmic bytes per
    item (SURVEY 8(d)): train forward 6 184 B, + 3 072 B of injected uniforms for Gumbel; backward 9 244 B."""
    T, beta = 0.2, 0.25
    xg = x.detach().clone().requires_grad_(True)
    cg = [c.detach().clone().requires_grad_(True) for c in cbs]
    us = [torch.rand(N_ITEMS, K, device="cuda") for _ in range(L)]
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))

    def rot_fwd():
        return ops.RqChainFunction.apply(xg, ops.MODE_ROTATION, beta, True, *cg)

    def rot_fb():
        e, _n, _i, loss = rot_fwd()
        (e.sum() + loss.sum()).backward()

    def gum_fwd():
        res, tot, loss = xg, 0, 0
        for l in range(L):
            emb, _ids, ls = ops.GumbelQuantizeFunction.apply(res, cg[l], us[l], T, beta)
            res, tot, loss = res - emb, tot + emb, loss + ls
        return tot, loss

    def gum_fb():
        e, loss = gum_fwd()
        (e.sum() + loss.sum()).backward()

    out = {}
    with torch.no_grad():
        out["rotation_fwd_ms"] = _event_ms(torch, rot_fwd, n=5, warm=2)
        out["gumbel_fwd_ms"] = _event_ms(torch, gum_fwd, n=5, warm=2)
    out["rotation_fwd_bwd_ms"] = _event_ms(torch, rot_fb, n=5, warm=2)
    out["gumbel_fwd_bwd_ms"] = _event_ms(torch, gum_fb, n=5, warm=2)
    fwd_b, noise_b = 6184.0, 4.0 * K * L
    out["rotation_fwd_frac_of_hbm_roofline"] = N_ITEMS * fwd_b / (out["rotation_fwd_ms"] * 1e-3) / 1e9 / peak
    out["gumbel_fwd_frac_of_hbm_roofline"] = N_ITEMS * (fwd_b + noise_b) / (out["gumbel_fwd_ms"] * 1e-3) / 1e9 / peak
    out["gumbel_fwd_tflops_fp32_equivalent"] = 2 * 2.0 * N_ITEMS * D * K * L / (out["gumbel_fwd_ms"] * 1e-3) / 1e12
    out["note"] = ("fp32 I/O; rotation = tensor-core tokeniser (ids) + one streaming pass over the given ids (outputs, bit-identical to the "
                   "fused CUDA-core chain) + one backward launch; Gumbel = per level "
                   "split-precision tensor-core GEMMs x.C^T and W.C + row kernels; compute-bound, not HBM-bound: the fractions "
                   "say how far from the byte floor the FLOPs keep these paths")
    return {"items": N_ITEMS, **out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--path", default="auto", choices=["auto", "tc", "simt"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from rq_vae_recommender_b200 import ops
    from rq_vae_recommender_b200 import parallel

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    x_h, cbs_h = make_problem(N_ITEMS, seed=1234 + rank)          # every rank: its own 64K-item shard
    x = torch.from_numpy(x_h).cuda()
    cbs = [torch.from_numpy(c).cuda() for c in cbs_h]
    use_tc = args.path == "tc" or (args.path == "auto" and ops.tc_supported(D, K, L))
    tok = parallel.CorpusTokenizer(cbs, use_tc=use_tc)
    # one-time cost of the frozen-codebook state (not part of a step: the codebooks of a trained model do not change)
    prepare_ms = None
    if use_tc:
        ops.TcState(cbs)
        torch.cuda.synchronize()
        pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        pe0.record()
        ops.TcState(cbs)
        pe1.record()
        torch.cuda.synchronize()
        prepare_ms = pe0.elapsed_time(pe1)
    stats = torch.zeros(8, dtype=torch.int32, device="cuda") if use_tc else None

    def step():
        return tok.tokenize_device(x)

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # Clock sampling: the timed region is only K x ~0.4 ms, shorter than nvidia-smi's start-up + sampling period, so the
    # sampler is started first and the SAME step loop keeps the GPU under identical load until it is producing rows, and
    # again for a short continuation after the timed region: samples bracket the timed region under continuous load.
    with ClockSampler(local) as clocks:
        t_pre = time.perf_counter()
        while len(clocks.rows) < 2 and time.perf_counter() - t_pre < 3.0:
            for _ in range(50):
                ids = step()
            torch.cuda.synchronize()
        n_before = len(clocks.rows)
        for _ in range(max(args.warmup, 3)):
            ids = step()
        sync()
        l0 = ops.LAUNCHES
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
        ev[0].record()
        for i in range(args.steps):
            ids = step()
            ev[i + 1].record()
        sync()
        launches_timed = ops.LAUNCHES - l0
        t_post = time.perf_counter()
        while time.perf_counter() - t_post < 0.5:       # continuation of the same load (untimed) so rows land after it too
            for _ in range(50):
                step()
            torch.cuda.synchronize()
        n_after = len(clocks.rows)
    ops.LAUNCHES = l0 + launches_timed                  # gpu_launches counts the timed region only
    launches = ops.LAUNCHES - l0
    rerank = None
    if use_tc:                                          # re-rank rate of the deterministic margin (one extra untimed pass)
        stats.zero_()
        tok.tokenize_device(x, stats=stats)
        st_h = stats.cpu().tolist()
        rerank = {"rows_reranked": st_h[0], "candidates_rescored": st_h[1], "rows_with_3plus_candidates": st_h[2],
                  "fraction_of_row_levels": st_h[0] / float(N_ITEMS * L)}
    total_ms = ev[0].elapsed_time(ev[-1])
    per_step = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    t = torch.tensor([total_ms], device="cuda")
    per_rank_ms = [total_ms / args.steps]
    if world > 1:
        gathered = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(gathered, t)
        per_rank_ms = [float(g.item()) / args.steps for g in gathered]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    value = world * N_ITEMS * args.steps / (total_ms * 1e-3)

    # ---- end to end through the host API: pinned host rows in, host ids out, copies inside the timed region
    xh_pinned = torch.from_numpy(x_h).pin_memory()
    for _ in range(2):
        tok.tokenize_host(xh_pinned)
    sync()
    e2e_steps = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ids_host = tok.tokenize_host(xh_pinned)
    sync()
    e2e_s = torch.tensor([time.perf_counter() - t0], device="cuda")
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = world * N_ITEMS * e2e_steps / float(e2e_s.item())
    # plain pinned host->device copy of the same batch: the ceiling any host-fed path has on this box
    xd_tmp = torch.empty_like(x)
    xd_tmp.copy_(xh_pinned, non_blocking=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(3):
        xd_tmp.copy_(xh_pinned, non_blocking=True)
    torch.cuda.synchronize()
    h2d_gbs = 3 * x_h.nbytes / (time.perf_counter() - t0) / 1e9
    del xd_tmp
    c3 = run_c3(world, rank, cbs if rank == 0 else [torch.from_numpy(c).cuda() for c in make_problem(8192, seed=1234)[1]],
                torch, dist, ops, parallel) if world > 1 else None

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
        kern_ms = float(np.mean(per_step))
        achieved = algorithmic_bytes(N_ITEMS) / (kern_ms * 1e-3) / 1e9
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "per_gpu_items": N_ITEMS,
                       "kernel": ("rq_tcx_kernel: tcgen05 fp16 filter (deterministic margin) + exact fp32 re-rank" if use_tc
                                  else "fp32 CUDA-core fused chain"),
                       "api": "parallel.CorpusTokenizer -> ops.rq_tokenize_tc with a prepared state: the routing RqVae.tokenize / "
                              "SemanticIdTokenizer.precompute_corpus_ids use (ops.rq_tokenize_auto)",
                       "ms_per_step_per_rank": per_rank_ms,
                       "parallelism": f"items sharded over {world} GPU(s), no data-path collective",
                       "l2": "input batch (201 MB) exceeds the 126 MB L2; no flush between steps"},
            "clocks": dict(clocks.summary(), note=("sampled at 100 ms over pre-load + warm-up + timed region + 0.5 s "
                                                  "continuation of the same step loop (timed region itself: "
                                                  f"{total_ms:.1f} ms); rows before/after the timed region: {n_before}/{n_after - n_before}")),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(x_h.nbytes),
                    "d2h_bytes_per_step": int(N_ITEMS * L * 8), "steps": e2e_steps,
                    "h2d_copy_gbs_measured": h2d_gbs,
                    "h2d_bound_items_per_sec": world * h2d_gbs * 1e9 / (4 * D)},
            "gpu_launches": launches,
            "prepare_ms": prepare_ms,
            "rerank": rerank,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
                         "frac": achieved / peak_gbs, "traffic": tok.measured_traffic_bytes(),
                         "traffic_source": "static: dram__bytes_read.sum + dram__bytes_write.sum of the committed ncu --set full "
                                           "capture of this kernel at this shape (profiles/r2_tcx_ncu_summary.csv), not measured in this run",
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "6650 GB/s (of fallback)",
                         "kernel_ms": kern_ms, "algorithmic_bytes": algorithmic_bytes(N_ITEMS)},
        }
        if c3 is not None:
            out["c3"] = c3
        if world == 1:
            for name, fn in (("c2", lambda: run_c2(x, cbs, torch, ops)), ("pipeline", lambda: run_pipeline(torch, ops)),
                             ("c4", lambda: run_c4(x, cbs, torch, ops))):
                try:
                    out[name] = fn()
                except Exception as e:        # an auxiliary record must never take the headline line down
                    out[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
        if world == 1 and not args.no_cpu_baseline:
            v, threads, sample = cpu_port_items_per_sec(x_h, cbs_h)
            out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample}
        # sanity: the timed result is the real answer
        from oracle import rq_oracle as O
        chk = O.rq_tokenize(x_h[:512], cbs_h)
        agree = float((ids[:512].cpu().numpy() == chk).all(1).mean())
        out["config"]["oracle_agreement_512"] = agree
        print(json.dumps(out))
    if args.dump_outputs:                               # `ids` is still the last timed step's result
        dump_outputs(args.dump_outputs, {"ids" if world == 1 else f"ids_rank{rank}": ids})
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
