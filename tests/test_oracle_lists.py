"""CPU (-m "not gpu"): the oracle's BaseType::lrt(specific_bases) over ordered candidate lists (bvo_site_list,
tests/oracle_lists.c, built on oracle/bv_oracle.c) is pinned
  * to the oracle's own lrt() (bvo_site) for the list A,C,G,T, bit for bit, on the golden sites and on random tiles,
  * to its population-group call (bvo_group_site) for [REF, ALT...] lists over planes masked to one group,
  * to the compiled reference's own lrt(basecombination) group outputs in the committed tests/golden/calls_*.npz.
"""
import glob
import os

import numpy as np
import pytest

from oracle import loader as L
from tests import oracle_lists as OL
from tests import util

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
LRT_FLAGS = 0x04 | 0x10 | 0x40 | 0x80   # ZERO_SUBSET, NEAR_LRT, EM_MAXITER, LRT_TIE


def same_f64(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return (a.view(np.uint64) == b.view(np.uint64)) | (np.isnan(a) & np.isnan(b))


def acgt_lists(S):
    return np.tile(np.arange(4, dtype=np.uint8), (S, 1))


def assert_list_equals_site(lrt, recs, label):
    for f in ("n_alt", "n_active", "flags", "em_calls"):
        assert (lrt[f] == recs[f]).all(), f"{label}: {f} differs at {np.nonzero(lrt[f] != recs[f])[0][:10]}"
    assert (lrt["alt"] == recs["alt"]).all(), f"{label}: alt differs"
    assert same_f64(lrt["af"], recs["af"]).all(), f"{label}: af differs"
    for a, b in (("qual", "qual"), ("chi2", "chi2"), ("fs", "fs_vcf")):
        assert same_f64(lrt[a], recs[b]).all(), f"{label}: {a} differs at {np.nonzero(~same_f64(lrt[a], recs[b]))[0][:10]}"


def golden_site_files():
    return sorted(glob.glob(os.path.join(GOLDEN_DIR, "sites_minaf_*.npz")))


@pytest.mark.parametrize("path", golden_site_files(), ids=os.path.basename)
@pytest.mark.parametrize("mode", [0, 1])
def test_acgt_list_is_lrt_on_golden_sites(oracle_lib, path, mode):
    z = np.load(path)
    N, maf = int(z["n_samples"]), float(z["min_af"])
    S = z["base"].shape[0]
    recs = L.oracle_tile(z["base"], z["qual"], z["strand"], z["ref_base"], N, maf, mode)
    lrt = OL.oracle_lists(z["base"], z["qual"], z["strand"], z["ref_base"], acgt_lists(S), N, maf, mode)
    assert_list_equals_site(lrt, recs, os.path.basename(path))


@pytest.mark.parametrize("mode", [0, 1])
def test_acgt_list_is_lrt_on_random_tiles(oracle_lib, mode):
    rng = np.random.default_rng(2026 + mode)
    for (S, N, cov, qlo, qhi, other, indel, bad, maf) in [
        (200, 40, 0.9, 0, 40, 0.05, 0.05, 0.0, 0.01),      # phred-0 reads, other / indel cells
        (150, 300, 0.3, 2, 60, 0.01, 0.02, 0.01, 0.05),    # bad strand symbols
        (60, 1200, 0.6, 10, 41, 0.0, 0.0, 0.0, 0.01),
        (100, 64, 0.8, 0, 93, 0.02, 0.0, 0.0, 0.2),
    ]:
        b, q, s, r = util.random_tile(rng, S, N, cov, qlo, qhi, other=other, indel=indel, bad_strand=bad)
        recs = L.oracle_tile(b, q, s, r, N, maf, mode)
        lrt = OL.oracle_lists(b, q, s, r, acgt_lists(S), N, maf, mode)
        assert_list_equals_site(lrt, recs, f"N={N} maf={maf}")


def mask_to_group(base, qual, strand, sample_group, g):
    N = sample_group.shape[0]
    out = base.copy(), qual.copy(), strand.copy()
    off = np.nonzero(sample_group != g)[0]
    out[0][:, off] = 5
    out[1][:, off] = 0
    out[2][:, off] = 2
    out[0][:, N:] = 5
    return out


def group_lists(ref_base, recs):
    lists = np.full((len(ref_base), 4), OL.LIST_END, np.uint8)
    for s in range(len(ref_base)):
        order = L._group_order(int(ref_base[s]), recs[s])
        lists[s, :len(order)] = order
    return lists


def test_ref_alt_lists_are_the_group_call(oracle_lib):
    rng = np.random.default_rng(11)
    for (S, N, cov, G) in [(200, 80, 0.7, 3), (60, 600, 0.3, 5)]:
        b, q, s, r = util.random_tile(rng, S, N, cov, 0, 60, other=0.02, indel=0.02)
        grp = util.random_groups(rng, N, G)
        recs = L.oracle_tile(b, q, s, r, N, 0.01, 0)
        lists = group_lists(r, recs)
        _, want = L.oracle_calls(b, q, b, np.zeros(b.shape, np.uint16), r, N, recs, grp, G, 0.01, 0)
        called = np.nonzero(recs["n_alt"] > 0)[0]
        for g in range(G):
            mb, mq, ms = mask_to_group(b, q, s, grp, g)
            got = OL.oracle_lists(mb[called], mq[called], ms[called], r[called], lists[called], N, 0.01, 0)
            w = want[:, g]
            assert (got["n_alt"] == w["n_alt"]).all() and (got["alt"] == w["alt"]).all(), f"N={N} group {g}: ALT differs"
            assert same_f64(got["af"], w["af"]).all(), f"N={N} group {g}: AF differs"
            assert ((got["flags"] & (LRT_FLAGS | 0x02)) == (w["flags"] & (LRT_FLAGS | 0x02))).all(), f"N={N} group {g}: flags differ"


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN_DIR, "calls_*.npz"))), ids=os.path.basename)
def test_ref_alt_lists_reproduce_the_reference_group_calls(oracle_lib, path):
    """The reference's own lrt([REF, ALT...]) outputs (make_golden_calls.py) from bvo_site_list over group-masked planes."""
    z = np.load(path)
    N, G, maf = int(z["n_samples"]), int(z["n_groups"]), float(z["min_af"])
    for mode, key in ((0, "int"), (1, "dbl")):
        recs = z["recs_" + key].view(L.SITE_OUT_DTYPE)
        called = np.nonzero(recs["n_alt"] > 0)[0]
        want = z["groups_" + key].view(L.GROUP_OUT_DTYPE).reshape(len(called), G)
        lists = group_lists(z["ref_base"], recs)[called]
        for g in range(G):
            mb, mq, ms = mask_to_group(z["base"], z["qual"], z["strand"], z["sample_group"], g)
            got = OL.oracle_lists(mb[called], mq[called], ms[called], z["ref_base"][called], lists, N, maf, mode)
            w = want[:, g]
            label = f"{os.path.basename(path)} mode {mode} group {g}"
            assert (got["n_alt"] == w["n_alt"]).all() and (got["alt"] == w["alt"]).all(), f"{label}: ALT differs"
            assert same_f64(got["af"], w["af"]).all(), f"{label}: AF differs"


def test_invalid_and_empty_lists(oracle_lib):
    b, q, s, r, N = L.planes_from_reads([("A", [("A", 30, "+")] * 7 + [("G", 30, "-")] * 3)])
    for bad in ([0, 0, OL.LIST_END, OL.LIST_END], [0, 4, OL.LIST_END, OL.LIST_END], [7, OL.LIST_END, 0, 0]):
        with pytest.raises(AssertionError):
            OL.oracle_lists(b, q, s, r, np.array([bad], np.uint8), N)
    empty = OL.oracle_lists(b, q, s, r, np.full((1, 4), OL.LIST_END, np.uint8), N)
    assert empty.tobytes() == bytes(64)
