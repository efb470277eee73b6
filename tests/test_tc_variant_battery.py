"""CPU check that the tile-shape battery of tests/tc_variant_child.py (run on the GPU by tests/test_gpu_tc_variants.py) reaches
every case it exists for, at the 148 SMs of a B200.  The tile arithmetic of tcx_run (csrc/rq_tcx.cu) and the build choice of
rqb200_tokenize_tc_run (csrc/rq_tc.cu) are restated in tc_variant_child.py; the constants and formulas are matched against
the CUDA sources here, so an edit to either side that breaks the restatement fails this file."""
import os
import re

import pytest

import tc_variant_child as C

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "rq_vae_recommender_b200", "csrc")
SMS = 148


def src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def define(text, name):
    m = re.search(rf"^#define\s+{name}\s+(\d+)\b", text, re.M)
    assert m, f"#define {name} not found"
    return int(m.group(1))


def tile_constants():
    """{rows per CTA: TX_NT} from the two builds' #define blocks, after checking the rest of the restatement."""
    tcx, tcx96, common, tc = src("rq_tcx.cu"), src("rq_tcx96.cu"), src("tc_common.cuh"), src("rq_tc.cu")
    assert define(tcx, "TX_R") == 64 and define(tcx96, "TX_R") == 96
    assert re.search(r"#include\s+\"rq_tcx\.cu\"", tcx96), "rq_tcx96.cu no longer compiles rq_tcx.cu at TX_R = 96"
    assert {r: 2 * r for r in (64, 96)} == C.PAIR_ROWS
    assert re.search(r"^#define\s+TX_PR\s+\(2 \* TX_R\)", tcx, re.M), "pair tile is no longer 2 * TX_R rows"
    assert define(common, "TC_KC") == 64 and define(common, "TC_MAX_D") == 768
    assert re.search(r"p\.nkc\s*=\s*D\s*/\s*TC_KC;", tcx)
    assert re.search(r"p\.ntiles\s*=\s*\(B\s*\+\s*TX_PR\s*-\s*1\)\s*/\s*TX_PR;", tcx)
    assert re.search(r"nclusters\s*=\s*p\.ntiles\s*<\s*sm_count\s*/\s*2\s*\?\s*p\.ntiles\s*:\s*sm_count\s*/\s*2;", tcx)
    assert re.search(r"u_first\s*=\s*\(int\)\(blockIdx\.x\s*>>\s*1\),\s*u_step\s*=\s*\(int\)\(gridDim\.x\s*>>\s*1\)", tcx), \
        "pair tiles are no longer dealt round-robin to the CTA pairs"
    assert re.search(r"force\s*\?\s*force\s*==\s*96\s*:\s*\(int64_t\)B\s*>\s*128ll\s*\*\s*\(sm_count\s*/\s*2\)", tc), \
        "the default tile-shape switch of rqb200_tokenize_tc_run changed"
    m = re.search(r"#if TX_R == 64\n(.*?)#else\n(.*?)#endif", tcx, re.S)
    assert m, "tile-shape #if block of rq_tcx.cu not found"
    return {64: define(m.group(1), "TX_NT"), 96: define(m.group(2), "TX_NT")}


def test_restated_tile_arithmetic_matches_the_sources():
    nt = tile_constants()
    assert nt == {64: 4, 96: 2}, nt
    pairs = SMS // 2
    assert C.default_rows(128 * pairs, SMS) == 64 and C.default_rows(128 * pairs + 1, SMS) == 96
    assert C.tiles(64, 1, SMS) == (1, 1, 1)
    assert C.tiles(64, 128 * pairs, SMS) == (pairs, pairs, 1)
    assert C.tiles(64, 128 * pairs + 1, SMS) == (pairs + 1, pairs, 2)
    assert C.tiles(96, 65536, SMS) == (342, pairs, 5)


@pytest.fixture(scope="module")
def battery():
    b = C.battery(SMS)
    names = [p.name for p in b]
    assert len(set(names)) == len(names), "problem names must be unique (they key the child's outputs)"
    return b


def test_battery_covers_tiles_per_pair_of_both_builds(battery):
    """Each build runs 1 .. TX_NT + 1 tiles on every CTA pair and 2 .. TX_NT + 2 tiles with some pairs idle in the last round
    (TX_NT of the deeper build): every TMEM, exchange and row-statistics ring wraps, with and without a partial last round.
    (With one tile per pair the grid shrinks to the tile count: that last round is never partial.)"""
    nmax = max(tile_constants().values())
    for R in (64, 96):
        full, partial = set(), set()
        for p in battery:
            ntiles, nclusters, per_pair = C.tiles(R, p.B, SMS)
            (full if ntiles % nclusters == 0 else partial).add(per_pair)
        for t in range(1, nmax + 2):
            assert t in full, f"{R}-row build: no problem runs {t} tiles on every CTA pair (B = {t * C.PAIR_ROWS[R] * (SMS // 2)})"
        for t in range(2, nmax + 3):
            assert t in partial, f"{R}-row build: no problem runs {t} tiles per CTA pair with a partial last round"
    assert max(C.tiles(64, p.B, SMS)[2] for p in battery) > 100, "no problem gives the 64-row build > 100 tiles per pair"


def test_battery_covers_every_width(battery):
    direct = {p.D // 64 for p in battery if p.direct}
    for nkc in range(1, 768 // 64 + 1):
        assert nkc in direct, f"no problem calls the kernel directly at nkc = {nkc} (D = {64 * nkc})"
    padded = {C.padded_dim(p.D) // 64 for p in battery if not p.direct}
    for nkc in (1, 2, 11):
        assert nkc in padded, f"no problem reaches nkc = {nkc} through the zero-padding path of TcState"
    for p in battery:
        assert p.ldx is None or (p.direct and p.ldx > p.D and p.ldx % 4 == 0), p
    assert sum(p.ldx is not None for p in battery) >= 3, "too few problems with a padded row stride"


def test_battery_covers_levels(battery):
    have = {(p.D, p.L) for p in battery}
    for D in (64, 768):
        for L in (1, 8):
            assert (D, L) in have, f"no problem at D = {D}, L = {L}"


def test_battery_covers_tails_in_every_row_group(battery):
    """A partial last pair tile whose last row falls in each 32-row scan group, for both builds."""
    for R, P in C.PAIR_ROWS.items():
        groups = {(p.B % P - 1) // 32 for p in battery if p.B % P}
        for g in range(P // 32):
            assert g in groups, f"{R}-row build: no partial pair tile ends in rows [{32 * g}, {32 * g + 32})"


def test_battery_covers_switch_and_special_rows(battery):
    Bs = {p.B for p in battery}
    switch = 128 * (SMS // 2)
    assert switch in Bs and switch + 1 in Bs, "the default tile-shape switch point and the row above it"
    special = [p for p in battery if p.kind == "special"]
    assert max((p.B for p in special), default=0) > 2 * max(C.PAIR_ROWS.values()), "special rows in > 2 pair tiles of both builds"
    for p in special:
        rows = C.special_rows(p.B)
        assert set(rows.values()) == set(C.SPECIAL_KINDS) and p.B - 1 in rows
        for P in C.PAIR_ROWS.values():
            for t0 in range(0, p.B - P, P):
                for h in (0, P // 2):
                    for r in (0, 31, 32, 63):
                        assert t0 + h + r in rows, f"{p.name}: no special row at local row {r} of half {h} of tile {t0}"
    fams = {p.kind[4:] for p in battery if p.kind.startswith("adv:")}
    import tc_filter_model as M
    assert fams == set(M.ADVERSARIAL_KINDS)
    assert any(p.kind == "judge" for p in battery)
