"""Both tile shapes of the tensor-core tokeniser (64 and 96 rows per CTA, csrc/rq_tcx.cu / rq_tcx96.cu) on the battery of
tests/tc_variant_child.py: every width, tail, tile count per CTA pair and level count, special rows at the tile seams,
adversarial rounding and the deep shapes.  `pytest -m gpu`.

RQB200_TC_ROWS is read once per process, so each configuration (the default choice by batch size, 64 forced, 96 forced) runs
in a child process of its own; the child records the raw outputs and this module asserts on them:
  per configuration  every row below B holds an id in [0, 256) and every guard row is still -1; x and the prepared state are
                     unchanged; 0 <= stats[2] <= stats[0] <= B L (and stats[1] >= 2 stats[0] on finite inputs); the ids are the
                     exact CUDA-core kernel's (and, up to B = 20 000, the fp32 oracle's) under the near-tie protocol of parity.py,
                     with at most max(2, B / 2000) near ties outside the adversarial families
  across them        identical input bytes, bit-identical ids and identical stats[0..2] (candidate sets, margins and the exact
                     re-rank are per-row functions of the prepared state: the tile geometry must not show)
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import tc_variant_child as C
from oracle import rq_oracle as O
from parity import assert_ids_match

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
CONFIGS = {"default": None, "r64": "64", "r96": "96"}
CHILD_TIMEOUT_S = 600
ORACLE_MAX_B = 20000


@pytest.fixture(scope="module")
def runs(tmp_path_factory):
    """{config: npz of the child's outputs}.  A child that fails or times out fails the module with its stderr."""
    out = {}
    tmp = tmp_path_factory.mktemp("tc_variants")
    for cfg, rows in CONFIGS.items():
        env = dict(os.environ)
        for k in ("RQB200_TC_ROWS", "RQB200_TC_TRACE", "RQB200_TC_PREFETCH"):
            env.pop(k, None)
        if rows is not None:
            env["RQB200_TC_ROWS"] = rows
        path = str(tmp / f"{cfg}.npz")
        cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.join(HERE, "tc_variant_child.py"), path]
        try:
            r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=CHILD_TIMEOUT_S)
        except subprocess.TimeoutExpired as e:
            pytest.fail(f"{cfg}: child timed out after {CHILD_TIMEOUT_S} s\n{e.stderr}")
        assert r.returncode == 0, f"{cfg}: child exited with {r.returncode}\n{r.stdout}\n{r.stderr}"
        print(f"[{cfg}] {r.stdout.strip()}")
        out[cfg] = np.load(path)
    return out


@pytest.fixture(scope="module")
def problems(runs):
    sm_count = torch.cuda.get_device_properties(0).multi_processor_count
    for cfg, z in runs.items():
        assert int(z["sm_count"]) == sm_count, cfg
    return C.battery(sm_count)


def test_children_tokenised_identical_inputs(runs, problems):
    for p in problems:
        shas = {cfg: str(z[p.name + "/sha"]) for cfg, z in runs.items()}
        assert len(set(shas.values())) == 1, f"{p.name}: input bytes differ between configurations {shas}"


def test_tile_shapes_return_identical_ids_and_stats(runs, problems):
    bad = []
    for p in problems:
        ref = runs["default"]
        for cfg in ("r64", "r96"):
            a, b = runs[cfg][p.name + "/ids"], ref[p.name + "/ids"]
            if not np.array_equal(a, b):
                rows = np.nonzero((a != b).any(1))[0] - (C.GUARD if p.direct else 0)
                bad.append(f"{p.name}: {cfg} vs default ids differ on {len(rows)} rows, first {rows[:8].tolist()}")
            sa, sb = runs[cfg][p.name + "/stats"], ref[p.name + "/stats"]
            if not np.array_equal(sa[:3], sb[:3]):
                bad.append(f"{p.name}: {cfg} stats {sa[:3].tolist()} vs default {sb[:3].tolist()}")
    assert not bad, "\n".join(bad)


def check_one(p, z, x, cbs, expect, exact, oracle):
    """Failures of one configuration on one problem (list of messages)."""
    bad = []
    ids = z[p.name + "/ids"]
    if p.direct:
        assert ids.shape == (p.B + 2 * C.GUARD, p.L)
        lo, hi = ids[:C.GUARD], ids[C.GUARD + p.B:]
        if (lo != -1).any() or (hi != -1).any():
            bad.append(f"guard rows written: before B {np.nonzero((lo != -1).any(1))[0].tolist()[:8]}, "
                       f"at or after B {(np.nonzero((hi != -1).any(1))[0]).tolist()[:8]} (offset from row B)")
        ids = ids[C.GUARD:C.GUARD + p.B]
    assert ids.shape == (p.B, p.L)
    out_of_range = np.nonzero(((ids < 0) | (ids >= C.K)).any(1))[0]
    if len(out_of_range):
        return bad + [f"{len(out_of_range)} rows hold no valid id (unwritten or garbage), first {out_of_range[:8].tolist()}: "
                      f"{ids[out_of_range[:2]].tolist()}"]
    for what in ("x", "state"):
        h = z[p.name + f"/{what}_hash"]
        if h[0] != h[1]:
            bad.append(f"the run modified {what}")
    s = z[p.name + "/stats"].astype(np.int64)
    if not (0 <= s[2] <= s[0] <= p.B * p.L) or s[3] != 0:
        bad.append(f"stats out of bounds: {s.tolist()} (B L = {p.B * p.L})")
    if np.isfinite(x).all() and s[1] < 2 * s[0]:
        bad.append(f"stats[1] = {s[1]} < 2 stats[0] = {2 * s[0]}: a re-ranked row has at least two candidates")
    if s[0] < expect.get("min_reranked", 0):
        bad.append(f"only {s[0]} rows re-ranked, expected >= {expect['min_reranked']}")
    if "level0_code" in expect and not (ids[:, 0] == expect["level0_code"]).all():
        bad.append(f"level-0 ids {np.unique(ids[:, 0]).tolist()}, expected all {expect['level0_code']}")
    if "copy_rows" in expect:
        got = ids[expect["copy_rows"], 0]
        if not np.array_equal(got, expect["copy_codes"]):
            bad.append(f"rows that copy a code: ids {got.tolist()} vs codes {expect['copy_codes'].tolist()}")
    keep = np.ones(p.B, bool)
    if "inf_rows" in expect:
        keep[expect["inf_rows"]] = False          # their neighbours must still match, row by row
    xk = x[keep]
    tie_budget = max(2, p.B // 2000)
    try:
        n_tie = assert_ids_match(ids[keep], exact[keep], xk, cbs, "vs exact kernel")
        # the re-rank sums a dot product over lanes and a butterfly, the exact kernel sequentially: on the adversarial families,
        # built to be dense in near ties, the two fp32 roundings part on many rows (each one still a float64 near tie)
        if not p.kind.startswith("adv:") and n_tie > tie_budget:
            bad.append(f"{n_tie} rows differ from the exact kernel on near ties (budget {tie_budget})")
    except AssertionError as e:
        bad.append(str(e).splitlines()[0])
    if oracle is not None:
        try:
            n_tie = assert_ids_match(ids[keep], oracle[keep], xk, cbs, "vs fp32 oracle")
            if p.kind == "rq" and n_tie > tie_budget:          # fp16-overflowing and adversarial rows tie the fp32 oracle more often
                bad.append(f"{n_tie} rows differ from the fp32 oracle on near ties (budget {tie_budget})")
        except AssertionError as e:
            bad.append(str(e).splitlines()[0])
    return bad


def test_each_tile_shape_against_exact_kernel(runs, problems):
    from rq_vae_recommender_b200 import ops
    bad = []
    for p in problems:
        x, cbs, expect = C.make_problem(p)
        exact = ops.rq_tokenize(torch.from_numpy(x).cuda(), [torch.from_numpy(c).cuda() for c in cbs]).cpu().numpy()
        oracle = None
        if p.B <= ORACLE_MAX_B:
            with np.errstate(all="ignore"):
                oracle = O.rq_tokenize(x, cbs)
        for cfg, z in runs.items():
            bad += [f"{p.name} [{cfg}] {m}" for m in check_one(p, z, x, cbs, expect, exact, oracle)]
    assert not bad, f"{len(bad)} failures:\n" + "\n".join(bad[:60])
