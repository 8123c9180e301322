"""-m gpu: K4 (K4a bv_hist_kernel, K4b bv_em_task_kernel / bv_em_iter_kernel) at its capacity edges, against the oracle.

  1. Bin counts on both sides of the edges where the kernels change how they hold a site's (base, phred) bins: more than
     kStageBins = 96 (K4b and bv_em_iter_kernel read them from the pool in global memory instead of shared memory), more
     than kSmemBins = 160 (K4a's compaction goes through the per-warp spill rows), up to kMaxBins = 480 (every base code
     0..4 at every phred 0..95); with 1-4 active alleles, short and long rows (K4a's two shapes), tiles on both sides of
     kG4MaxTasks (four lanes or one lane per EM task), both EM modes, dense and sparse tiles.
  2. Tiles that fill each part of a slot's EM scratch (bin pool, pair tasks, triple tasks) at the smallest context they fit
     in: the records must be the same bytes as in a context eight times as large, and as in a second run.

Every tile is built with an exact set of bins per site, and the bin counts and active sets are checked on the host before the
tile is run, so that a tile cannot drift off the edge it is meant to test."""
import numpy as np
import pytest

import basevar_b200 as bv
from oracle import loader as L
from tests import util

pytestmark = pytest.mark.gpu
MIN_AF = 0.05                # high enough for inactive alleles of 96 bins in a 5,000-read row
EDGE_BINS = [1, 2, 95, 96, 97, 159, 160, 161, 255, 376, 470, 480]
G4_MAX_TASKS = 12288         # bv_em_kernels.cuh kG4MaxTasks


def feasible(nb, k, N):
    return k <= nb <= util.max_bins(k, N, MIN_AF)


def check_oracle(got, want, label):
    ie, fe, flips = util.compare_records(got, want)
    msg = ""
    if len(ie):
        msg += f"\n{label}: {len(ie)} sites differ in exact fields, first {ie[:5].tolist()}:\n got  {util.describe(got[ie[0]])}\n want {util.describe(want[ie[0]])}"
    if len(fe):
        msg += f"\n{label}: {len(fe)} sites out of tolerance, first {fe[:5].tolist()}:\n got  {util.describe(got[fe[0]])}\n want {util.describe(want[fe[0]])}"
    assert not msg, msg
    assert len(flips) <= 2, f"{label}: {len(flips)} threshold / tie flips"
    util.report_flips(label, got, want, flips)


def run_all_forms(eng, b, q, s, r, N):
    """Records of the tile as dense planes, as BV_CELLS_U32 and as BV_CELLS_U16 cells; the three must be the same bytes."""
    dense = eng.call_host(b, q, s, r, N)
    cells, _, start = bv.dense_to_sparse(b, q, s, N)
    u32 = eng.call_sparse(cells, start, r, N)
    words, _, start16 = bv.sparse_encode16(cells, start)
    u16 = eng.call_sparse(words, start16, r, N)
    assert u32.tobytes() == dense.tobytes(), "BV_CELLS_U32 tile differs from the dense tile"
    assert u16.tobytes() == dense.tobytes(), "BV_CELLS_U16 tile differs from the dense tile"
    return dense


@pytest.fixture(scope="module")
def engine(built_lib):
    # room for every tile below without filling the EM scratch (8,192 sites: 524,288 pool bins, 17,408 / 8,704 / 4,352 task slots)
    eng = bv.BaseTypeEngine(device=0, max_samples=5000, max_sites=8192, n_slots=2, min_af=MIN_AF)
    yield eng
    eng.close()


@pytest.mark.parametrize("abs_mode", [0, 1])
@pytest.mark.parametrize("lanes", ["g4", "g1"])
@pytest.mark.parametrize("N", [1000, 5000])
def test_bin_count_edges_vs_oracle(engine, N, lanes, abs_mode):
    rng = np.random.default_rng(N + (lanes == "g1"))
    shape = [(nb, k) for nb in EDGE_BINS for k in range(1, 5) if feasible(nb, k, N) for _ in range(2)]
    if N == 5000:   # the long rows hold every bin count at 2, 3 and 4 active alleles
        assert {(nb, k) for nb, k in shape if k >= 2} == {(nb, k) for nb in EDGE_BINS for k in (2, 3, 4) if nb >= k}
    if lanes == "g1":   # enough 4-allele sites of 20-90 bins to pass kG4MaxTasks
        shape += [(int(rng.integers(20, 91)), 4) for _ in range(G4_MAX_TASKS // 11 + 40)]
    shape = [shape[i] for i in rng.permutation(len(shape))]
    b, q, s, r = util.binned_tile(rng, shape, N, MIN_AF)
    nb, k = np.array(shape).T
    assert np.array_equal(util.bin_counts(b, q, N), nb)
    assert np.array_equal(util.active_counts(b, N, MIN_AF), k)
    n_tasks = sum(util.EM_TASKS[x] for x in k)
    assert (n_tasks > G4_MAX_TASKS) == (lanes == "g1"), n_tasks
    engine.set_params(min_af=MIN_AF, abs_mode=abs_mode)
    got = run_all_forms(engine, b, q, s, r, N)
    want = L.oracle_tile(b, q, s, r, N, MIN_AF, abs_mode)
    check_oracle(got, want, f"em-edges N={N} {lanes} abs={abs_mode}")
    deep = nb > 160
    assert (got["n_alt"][deep] > 0).sum() > 20 and (got["em_calls"][deep] >= 3).sum() > 20


# Three tiles, each of which fills a different part of the EM scratch of a context with max_sites = S first, under the
# sizing of the parent design (64 pool bins and 2 / 1 / 0.5 pair / triple / quad task slots per site):
#   pool:    2,048 sites, 2 active alleles, 300-480 bins       (about 800,000 bins against 64 S + 4,096)
#   pairs:   4,096 sites, 3 active alleles, <= 20 bins          (3 S pair tasks against 2 S + 1,024)
#   triples: 4,096 sites, 4 active alleles, <= 20 bins          (4 S triple tasks against S + 512)
SCRATCH_SHAPES = {"pool": (2048, 5000, 2, 300, 480), "pairs": (4096, 64, 3, 3, 20), "triples": (4096, 64, 4, 4, 20)}


@pytest.mark.parametrize("abs_mode", [0, 1])
@pytest.mark.parametrize("name", list(SCRATCH_SHAPES))
def test_scratch_capacity_does_not_change_records(built_lib, name, abs_mode):
    S, N, k, lo, hi = SCRATCH_SHAPES[name]
    rng = np.random.default_rng(17 + k)
    shape = [(int(x), k) for x in rng.integers(lo, hi + 1, S)]
    b, q, s, r = util.binned_tile(rng, shape, N, MIN_AF)
    assert np.array_equal(util.bin_counts(b, q, N), [x for x, _ in shape])
    assert (util.active_counts(b, N, MIN_AF) == k).all()
    runs = {}
    for label, max_sites in (("tight", S), ("ample", 8 * S), ("repeat", S)):
        eng = bv.BaseTypeEngine(device=0, max_samples=N, max_sites=max_sites, n_slots=1, min_af=MIN_AF, abs_mode=abs_mode)
        try:
            runs[label] = eng.call_host(b, q, s, r, N)
        finally:
            eng.close()
    for label in ("ample", "repeat"):
        diff =np.nonzero((runs[label].view(np.uint8).reshape(S, -1) != runs["tight"].view(np.uint8).reshape(S, -1)).any(axis=1))[0]
        assert len(diff) == 0, f"{name} abs={abs_mode}: {len(diff)} records of the {label} run differ from the tight run, first sites {diff[:10].tolist()}"
    got = runs["tight"]
    # the deep rows: a spot check of 256 sites; the short ones: every site
    idx = np.sort(rng.choice(S, 256, replace=False)) if N > 1000 else np.arange(S)
    want = L.oracle_tile(np.ascontiguousarray(b[idx]), np.ascontiguousarray(q[idx]), np.ascontiguousarray(s[idx]), r[idx].copy(), N, MIN_AF, abs_mode)
    check_oracle(got[idx], want, f"em-scratch {name} abs={abs_mode}")
    assert (got["em_calls"] >= 2).sum() > S // 2
