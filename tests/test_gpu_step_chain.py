"""-m gpu: the kernels of a tile chained with programmatic dependent launch against the same kernels run one after the other.

Unprofiled tiles launch K2..KF with programmatic stream serialization (a kernel's prologue overlaps the tail of the kernel before
it); profiled tiles (bv_set_profiling) launch them plainly, with events between them.  Each tile below runs once each way: the
records -- for compact tiles, the records they expand to -- must be the same bytes, and so must the number of launches.
The shapes cover every branch of the chain: both K1 / K4a row shapes around kLongRowSamples, both EM convergence tests (with and
without bv_em_iter_kernel), tiles where K3 or K4 has nothing to do, a tile smaller than one CTA, K2 over more sites than its
grid takes in one pass, and sparse tiles through K0 with compact results."""
import numpy as np
import pytest

import basevar_b200 as bv
from basevar_b200 import capi
from oracle import loader as L
from tests import util

pytestmark = pytest.mark.gpu


def _twice(eng, run):
    """run() unprofiled (chained) and profiled (serialised): (result, launches) of each."""
    out = []
    for prof in (False, True):
        eng.set_profiling(prof)
        l0 = eng.launch_count
        r = run()
        out.append((r, eng.launch_count - l0))
    eng.set_profiling(False)
    return out


def _dense(S, N, abs_mode=0, seed=1, edit=None, **kw):
    model = bv.synth.make_model(seed=seed, **kw)
    b, q, s, _, r = bv.synth_fill_host(model, 0, S, N)
    if edit is not None:
        edit(b, q, s, r, N)
    maf = bv.cli_min_af(0.01, N)
    eng = bv.BaseTypeEngine(device=0, max_samples=N, max_sites=S, n_slots=2, min_af=maf, abs_mode=abs_mode)
    try:
        (chained, l_c), (serial, l_s) = _twice(eng, lambda: eng.call_host(b, q, s, r, N))
    finally:
        eng.close()
    assert chained.tobytes() == serial.tobytes(), "records of the chained and the serialised launches differ"
    assert l_c == l_s
    return chained, (b, q, s, r, maf)


def _only_bound(b, q, s, r, N):
    """Every covered cell REF at phred 30, one read of another base per site: REF + one minor allele that K3's bound settles."""
    code = (np.arange(len(r)) & 3).astype(np.uint8)
    r[:] = np.frombuffer(b"ACGT", np.uint8)[code]
    b[:, :N] = code[:, None]
    q[:, :N] = 30
    s[:, :N] = np.arange(N, dtype=np.uint8) & 1
    b[:, 0] = (code + 1) & 3


@pytest.mark.parametrize("abs_mode", [0, 1])
@pytest.mark.parametrize(
    "name,S,N,kw",
    [
        ("C2-like", 20000, 1000, dict(coverage=0.1, variant_frac=0.05)),
        ("C5-like", 1500, 2000, dict(coverage=0.99326, variant_frac=0.5, multi_frac=0.5)),
        ("N4096", 600, 4096, dict(coverage=0.1, variant_frac=0.2, multi_frac=0.3)),
        ("N4097", 600, 4097, dict(coverage=0.1, variant_frac=0.2, multi_frac=0.3)),
        ("no-bound-sites", 3000, 60, dict(coverage=0.3, variant_frac=0.3)),   # depth < 22: K3 has nothing to do
        ("smaller-than-a-CTA", 100, 1000, dict(coverage=0.1, variant_frac=0.3)),
    ],
)
def test_chained_equals_serial(name, S, N, kw, abs_mode):
    _dense(S, N, abs_mode=abs_mode, seed=31 + N, **kw)


def test_chained_equals_serial_no_em_sites():
    rec, _ = _dense(2000, 40, seed=3, edit=_only_bound, coverage=1.0, variant_frac=0.0)
    assert (rec["n_alt"] == 0).all()
    assert ((rec["flags"] & capi.FLAG_LRT_BOUND) != 0).all(), "every site should be settled by K3's bound"


def test_chained_equals_serial_many_k2_passes():
    """More listed sites than K2's grid takes in one pass (2 CTAs per SM x 1,024 sites), checked against the oracle on a range."""
    rec, (b, q, s, r, maf) = _dense(400_000, 64, seed=9, coverage=1.0, variant_frac=0.9, multi_frac=0.5)
    n = 4000
    want = L.oracle_tile(b[:n], q[:n], s[:n], r[:n], 64, maf, 0)
    ie, fe, flips = util.compare_records(rec[:n], want)
    assert len(ie) == 0 and len(fe) == 0, f"{len(ie)} exact / {len(fe)} float mismatches vs the oracle"


@pytest.mark.parametrize("u16", [False, True])
def test_chained_equals_serial_sparse_compact(u16):
    S, N, tile = 30000, 1000, 8192
    model = bv.synth.make_model(seed=55, coverage=0.1, variant_frac=0.1, multi_frac=0.3)
    b, q, s, _, r = bv.synth_fill_host(model, 0, S, N)
    cells, _, st = bv.dense_to_sparse(b, q, s, N)
    if u16:
        cells, _, st = bv.sparse_encode16(cells, st)
    eng = bv.BaseTypeEngine(device=0, max_samples=N, max_sites=tile, n_slots=3, min_af=bv.cli_min_af(0.01, N))
    try:
        tiles = eng.sparse_tiles(cells, st, r, N, compact=True)

        def run():
            # (the full records of a compact tile are listed in an order that varies from run to run: compare the records they
            # expand to)
            out = np.zeros(S, bv.SITE_OUT_DTYPE)
            eng.run_sparse_tiles(tiles, compact=lambda s0, ns, briefs, full: eng.expand_compact(briefs, full, r[s0:s0 + ns],
                                                                                             out[s0:s0 + ns]))
            return out

        (chained, l_c), (serial, l_s) = _twice(eng, run)
    finally:
        eng.close()
    assert chained.tobytes() == serial.tobytes(), "compact results of the chained and the serialised launches differ"
    dense = bv.BaseTypeEngine(device=0, max_samples=N, max_sites=tile, n_slots=2, min_af=bv.cli_min_af(0.01, N))
    try:
        want = dense.call_host(b, q, s, r, N)
    finally:
        dense.close()
    assert chained.tobytes() == want.tobytes(), "compact sparse tiles and dense tiles give different records"
    assert l_c == l_s
