"""Problem battery of the tensor-core tokeniser's tile shapes, and the child process that runs it under one configuration.

`rqb200_tokenize_tc_run` (csrc/rq_tc.cu) picks the 64-row or the 96-row build of rq_tcx_kernel by batch size and reads
RQB200_TC_ROWS once per process, so tests/test_gpu_tc_variants.py starts this file once per configuration:

    python tests/tc_variant_child.py OUT.npz          (RQB200_TC_ROWS unset, =64 or =96 in the environment)

For every problem of `battery(sm_count)` the child builds the inputs from seeds, tokenises them and records the raw outputs:
the id buffer with its guard rows, stats[0..3], a sha1 of the inputs and hashes of x and of the prepared state taken before
and after the run.  The parent test does all the asserting.

`battery()` and `Problem` are plain Python (no CUDA, no torch): tests/test_tc_variant_battery.py checks on the CPU that the
sizes reach every tile-shape case they are meant to reach.
"""
import hashlib
import os
import sys
from typing import NamedTuple, Optional

import numpy as np

K = 256
GUARD = 64                      # id rows before and after the B rows the kernel may write, pre-filled with -1
PAIR_ROWS = {64: 128, 96: 192}  # rows per CTA pair tile of each build (TX_PR = 2 * TX_R)
SPECIAL_OFFSETS = (0, 31, 32, 63, 95)   # rows of a CTA's half of a pair tile: 32-row group edges of both builds
SPECIAL_KINDS = ("small", "large", "overflow", "zero", "copy", "inf")


class Problem(NamedTuple):
    name: str
    B: int
    D: int
    L: int
    seed: int
    kind: str = "rq"            # "rq" | "special" | "adv:<family of tc_filter_model>" | "judge"
    ldx: Optional[int] = None   # row stride in floats (None: D); > D puts NaN columns between the rows

    @property
    def direct(self) -> bool:
        """D a multiple of 64: the child calls the C entry point itself (guard rows); otherwise ops.rq_tokenize_tc pads."""
        return self.D % 64 == 0


def battery(sm_count: int):
    """Every problem, as a function of the SM count only."""
    pairs = sm_count // 2
    P = []
    # widths: every multiple of 64 (odd and even numbers of 64-wide k-chunks), a ragged B; a few with a padded row stride
    for D in range(64, 769, 64):
        P.append(Problem(f"width_D{D}", 1000 + D, D, 3, seed=D, ldx=D + 4 if D in (192, 448, 704) else None))
    for D in (1, 33, 100, 700):                                  # zero-padded to 64 / 64 / 128 / 704 by TcState
        P.append(Problem(f"padded_D{D}", 1000 + D, D, 3, seed=7 + D))
    # tails: the 32-row group, 96-row box, CTA and pair-tile edges of both builds
    for B in (1, 31, 32, 33, 63, 64, 65, 95, 96, 97, 127, 128, 129, 191, 192, 193, 255, 257, 383, 385):
        P.append(Problem(f"tail_B{B}", B, 128, 2, seed=3000 + B))
    # tiles per CTA pair: t of them with a partial last tile (-37) and t + 1 with one tile in the last round (+1)
    for R, widths in ((64, (64, 192, 128, 320, 256)), (96, (192, 128, 320, 64, 256))):
        for t in range(1, 6):
            for delta in (-37, 1):
                B = t * PAIR_ROWS[R] * pairs + delta
                P.append(Problem(f"tiles_r{R}_t{t}{delta:+d}", B, widths[t - 1], 3, seed=R * 100 + t * 10 + (delta > 0),
                                 ldx=widths[t - 1] + 68 if t == 3 else None))
    switch = 128 * pairs                                          # the default picks the 96-row build above this
    P.append(Problem("switch", switch, 256, 3, seed=41))
    P.append(Problem("switch+1", switch + 1, 256, 3, seed=42))
    # levels: the id-byte region and with it the codebook ring depth change with L
    for D in (64, 768):
        for L in (1, 2, 4, 5, 7, 8):
            P.append(Problem(f"levels_D{D}_L{L}", 1500 + 7 * L, D, L, seed=500 + D + L))
    # special rows at the tile seams of both builds, ~2.5 pair tiles
    P.append(Problem("special_D768", 485, 768, 3, seed=61, kind="special"))
    P.append(Problem("special_D128", 333, 128, 2, seed=62, kind="special", ldx=132))
    # adversarial rounding (tests/tc_filter_model.py) and the round-1 counterexample
    for fam in ("judge_r1", "sign_biased", "equal_magnitude", "code_parallel", "tiny_and_huge", "opposite_rounding"):
        P.append(Problem(f"adv_{fam}", 300, 768, 3, seed=5, kind="adv:" + fam))
    P.append(Problem("judge", 256, 768, 1, seed=5, kind="judge"))
    # deep: the benchmark shape, and > 100 tiles per pair on the 64-row build
    P.append(Problem("ns_65536x768", 65536, 768, 3, seed=1234, ldx=772))
    P.append(Problem("deep_2e20x64", 1 << 20, 64, 3, seed=2020))
    return P


# ---------------------------------------------------------------------------------------------------- tile arithmetic
def tiles(R: int, B: int, sm_count: int):
    """(pair tiles, CTA pairs launched, most tiles one pair runs) of the R-row build at B rows (tcx_run in csrc/rq_tcx.cu)."""
    ntiles = (B + PAIR_ROWS[R] - 1) // PAIR_ROWS[R]
    nclusters = min(ntiles, sm_count // 2)
    return ntiles, nclusters, -(-ntiles // nclusters)


def default_rows(B: int, sm_count: int) -> int:
    """Build the unforced rqb200_tokenize_tc_run picks (csrc/rq_tc.cu)."""
    return 96 if B > 128 * (sm_count // 2) else 64


def padded_dim(D: int) -> int:
    return -(-D // 64) * 64


# ---------------------------------------------------------------------------------------------------- problem data
def special_rows(B: int):
    """Row -> kind: offsets SPECIAL_OFFSETS of both CTA halves of every pair tile of both builds, and the last row."""
    rows = set()
    for P in PAIR_ROWS.values():
        for t0 in range(0, B, P):
            for h in (0, P // 2):
                rows.update(t0 + h + r for r in SPECIAL_OFFSETS if r < P // 2)
            rows.add(t0 + P - 1)
    rows = sorted(r for r in rows if r < B - 1) + [B - 1]
    n = len(SPECIAL_KINDS)          # shifted by one every round of kinds, so that each kind visits every kind of seam
    return {r: SPECIAL_KINDS[(i + i // n) % n] for i, r in enumerate(rows)}


def _live_codebooks(x, L, rs):
    """Codes = residual rows of a 4096-row sample plus gaussian jitter, walked level by level (every code attracts rows)."""
    sample = x[:4096].astype(np.float32)
    D = x.shape[1]
    res, cbs = sample.copy(), []
    for _ in range(L):
        idx = rs.choice(len(res), K, replace=len(res) < K)
        cb = (res[idx] + rs.standard_normal((K, D), dtype=np.float32) * np.float32(0.5 / np.sqrt(D))).astype(np.float32)
        cbs.append(cb)
        r64, c64 = res.astype(np.float64), cb.astype(np.float64)
        res = res - cb[np.argmin((c64 * c64).sum(1)[None, :] - 2.0 * (r64 @ c64.T), axis=1)]
    return cbs


def make_problem(p: Problem):
    """(x [B, D] fp32, codebooks, expectations).  Deterministic in p: every process builds identical bytes."""
    expect = {}
    if p.kind.startswith("adv:") or p.kind == "judge":
        import tc_filter_model as M
        fam = "judge_r1" if p.kind == "judge" else p.kind[4:]
        x, cbs = M.adversarial_problem(fam, D=p.D, L=p.L, n=p.B, seed=p.seed)
        if p.kind == "judge":
            expect["level0_code"] = 10          # fp32 / fp64 say code 10, the fp16 scores alone say 200
            expect["min_reranked"] = p.B
        return np.ascontiguousarray(x, np.float32), [np.ascontiguousarray(c, np.float32) for c in cbs], expect
    rs = np.random.default_rng(p.seed)
    n = max(p.B, 4096)
    x = rs.standard_normal((n, p.D), dtype=np.float32) * np.float32(1.0 / np.sqrt(p.D))     # rows of expected unit norm
    cbs = _live_codebooks(x, p.L, rs)
    x = np.ascontiguousarray(x[:p.B])
    if p.kind == "special":
        copy_rows, copy_codes, inf_rows = [], [], []
        for r, kind in special_rows(p.B).items():
            if kind == "small":
                x[r] *= np.float32(1e-3)
            elif kind == "large":
                x[r] *= np.float32(37.0)
            elif kind == "overflow":
                x[r] *= np.float32(1e6)             # fp16 overflow: every code is re-ranked exactly
            elif kind == "zero":
                x[r] = 0.0
            elif kind == "copy":
                x[r] = cbs[0][r % K]
                copy_rows.append(r)
                copy_codes.append(r % K)
            else:
                x[r, 5 % p.D] = np.inf
                inf_rows.append(r)
        expect.update(copy_rows=np.array(copy_rows), copy_codes=np.array(copy_codes), inf_rows=np.array(inf_rows))
    return x, cbs, expect


def input_sha(x, cbs) -> str:
    h = hashlib.sha1()
    for a in [x] + list(cbs):
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


# ---------------------------------------------------------------------------------------------------- child process
def _dev_sha(t) -> str:
    import torch
    return hashlib.sha1(t.detach().contiguous().view(-1).view(torch.uint8).cpu().numpy().tobytes()).hexdigest()


def run_problem(p: Problem, x, cbs):
    """Tokenise once under this process's configuration; returns the raw outputs."""
    import torch
    from rq_vae_recommender_b200 import _lib, ops
    B, D, L = p.B, p.D, p.L
    state = ops.TcState([torch.from_numpy(c).cuda() for c in cbs])
    stats = torch.zeros(4, dtype=torch.int32, device="cuda")
    if p.direct:
        ldx = p.ldx or D
        # x inside a buffer with NaN guard rows below B and NaN between the rows: the kernel must read neither
        xbuf = torch.full((B + GUARD, ldx), float("nan"), dtype=torch.float32, device="cuda")
        xbuf[:B, :D] = torch.from_numpy(x).cuda()
        ids = torch.full((GUARD + B + GUARD, L), -1, dtype=torch.int64, device="cuda")
        before = (_dev_sha(xbuf), _dev_sha(state.buf))
        torch.cuda.synchronize()
        rc = _lib.load().rqb200_tokenize_tc_run(xbuf.data_ptr(), ldx, B, state.buf.data_ptr(), D, K, L,
                                                ids[GUARD:].data_ptr(), stats.data_ptr(), torch.cuda.current_stream().cuda_stream)
        _lib.check(rc, f"tokenize_tc_run {p.name}")
    else:
        xbuf = torch.from_numpy(x).cuda()
        before = (_dev_sha(xbuf), _dev_sha(state.buf))
        torch.cuda.synchronize()
        ids = ops.rq_tokenize_tc(xbuf, state=state, stats=stats)
    torch.cuda.synchronize()
    after = (_dev_sha(xbuf), _dev_sha(state.buf))
    return dict(ids=ids.cpu().numpy(), stats=stats.cpu().numpy(), x_hash=np.array([before[0], after[0]]),
                state_hash=np.array([before[1], after[1]]))


def main(out_path: str) -> None:
    import time
    import torch
    sm_count = torch.cuda.get_device_properties(0).multi_processor_count
    out = {"sm_count": np.array(sm_count)}
    t0 = time.time()
    for p in battery(sm_count):
        x, cbs, _ = make_problem(p)
        r = run_problem(p, x, cbs)
        out[p.name + "/sha"] = np.array(input_sha(x, cbs))
        for k, v in r.items():
            out[p.name + "/" + k] = v
    np.savez(out_path, **out)
    print(f"{len(battery(sm_count))} problems, RQB200_TC_ROWS={os.environ.get('RQB200_TC_ROWS', '')}, "
          f"{time.time() - t0:.1f} s", flush=True)


if __name__ == "__main__":
    _here = os.path.dirname(os.path.abspath(__file__))
    for _p in (os.path.dirname(_here), os.path.join(_here, "golden"), _here):
        if _p not in sys.path:
            sys.path.insert(0, _p)
    main(sys.argv[1])
