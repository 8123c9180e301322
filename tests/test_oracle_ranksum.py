"""CPU (-m "not gpu"): the free-standing rank-sum helper of the tests (tests/oracle_ranksum.py: the classification rules of
ref_vs_alt_ranksumtest, the oracle's bvo_wilcoxon, the phred rule) is pinned to the compiled reference: truncated to int, it
gives the three rank sums of every called site of every tests/golden/calls_*.npz, in both abs modes, bit for bit.  The GPU
tests of bv_ranksum_test use it as their oracle."""
import glob
import os

import numpy as np
import pytest

from oracle import loader as L
from tests import oracle_ranksum as R

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN_DIR, "calls_*.npz"))), ids=os.path.basename)
def test_ranksum_helper_matches_golden_fixture(oracle_lib, path):
    z = np.load(path)
    N = int(z["n_samples"])
    for key in ("int", "dbl"):
        recs = z["recs_" + key].view(L.SITE_OUT_DTYPE)
        want = z["calls_" + key].view(L.CALL_OUT_DTYPE)
        sites, b, v, start, ref, mask = R.called_site_problems(z["base"], z["qual"], z["mapq"], z["rpr"], z["ref_base"], N, recs)
        assert np.array_equal(sites, want["site"]) and len(sites) > 0
        got = R.truncate(R.ranksum_batch(b, v, start, ref, mask)).reshape(-1, 3)
        for t, f in enumerate(("mq_rank_sum", "read_pos_rank_sum", "base_q_rank_sum")):
            bad = np.nonzero(got[:, t] != want[f])[0]
            assert len(bad) == 0, f"{os.path.basename(path)} {key} {f}: sites {sites[bad][:5]} got {got[bad, t][:5]} want {want[f][bad][:5]}"


def test_ranksum_helper_rules(oracle_lib):
    # SURVEY.md 8c: wilcoxon_ranksum_test({1,5,3,10,3,3,4,5},{6,7,2,2,8,9,10}) -> 0.271589; A = REF, C = ALT
    bases = np.array([0] * 8 + [1] * 7, np.uint8)
    values = np.array([1, 5, 3, 10, 3, 3, 4, 5, 6, 7, 2, 2, 8, 9, 10], np.int32)
    ph = R.ranksum_test(bases, values, ord("A"), 1 << 1)
    assert float(f"{10 ** (-ph / 10):.6g}") == 0.271589
    # a lowercase REF is upper-cased; a mask bit on REF changes nothing; N, other and indel codes are in neither class
    assert R.ranksum_test(bases, values, ord("a"), 0b0011) == ph
    noisy_b = np.concatenate([bases, np.array([4, 5, 6, 7], np.uint8)])
    noisy_v = np.concatenate([values, np.array([100, -5, 7, 0], np.int32)])
    assert R.ranksum_test(noisy_b, noisy_v, ord("A"), 1 << 1) == ph
    # REF N: every A/C/G/T base is judged by the mask alone, so no REF read here
    assert R.ranksum_test(bases, values, ord("N"), 0b0011) == 10000.0
    # every value tied: p == 1, and -10 log10(1) is -0.0
    tied = R.ranksum_test(bases, np.full(15, 7, np.int32), ord("A"), 1 << 1)
    assert tied == 0.0 and np.signbit(tied)
    # empty class
    assert R.ranksum_test(bases, values, ord("A"), 1 << 2) == 10000.0
