"""Shared helpers of the parity tests."""
import json
import os

import numpy as np

from basevar_b200 import capi

# Tolerance on floating-point outputs (AF, QUAL, FS): BASELINE.json's north_star allows 1e-6 relative; the
# histogram restatement only re-associates sums, so we hold the CUDA path to a much tighter bound.
RTOL = 1e-9
ATOL = 1e-12
# FS = -10*log10(p): the reference gets p from exp() of differences of lgamma(n) values, i.e. with an absolute error of
# about n * ulp(lgamma(n)) (1e-11 at n = 6000), so near p == 1 its FS carries absolute noise of that size; FS is
# printed with 6 decimals (std::to_string).
FS_ATOL = 1e-9


def close(a, b, rtol=RTOL, atol=ATOL):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    both_nan = np.isnan(a) & np.isnan(b)
    with np.errstate(invalid="ignore"):
        ok = np.abs(a - b) <= atol + rtol * np.abs(b)
    return ok | both_nan | (a == b)


def compare_records(got, want, check_diag=True, rtol=RTOL, soft_flags=None):
    """Compare CUDA records with oracle/reference records.

    Returns (exact_fail, float_fail, flips): integer fields (depths, strand tables) must always be bit-exact.
    A site whose call differs is a listed `flip`, not a failure, only in the two situations where the reference's
    own decision hangs on the last bits of a floating-point sum:
      * the LRT statistic sits on the threshold (BV_FLAG_NEAR_LRT), or
      * two candidate subsets tie (BV_FLAG_LRT_TIE): alleles with identical read multisets have equal likelihood;
        the reference's choice between them depends on rounding noise of its read-order sums.
    Which sites those are is decided by the ORACLE (oracle/bv_oracle.c computes both flags from its own statistics), never
    by the code under test: the mask is `want["flags"]`, or `soft_flags` (the oracle's flags for the same planes) when
    `want` comes from the compiled reference, whose records carry no such flags."""
    assert got.shape == want.shape
    n = got.shape[0]
    int_fail = np.zeros(n, bool)
    # a counted cell with a strand symbol other than +/- makes the reference throw (src/basetype.cpp:271-273):
    # for such sites only the flag and the depths are specified
    badst = ((got["flags"] | want["flags"]) & capi.FLAG_BAD_STRAND) != 0
    for f in ("depth", "depth_other"):
        x = got[f] != want[f]
        int_fail |= x.reshape(n, -1).any(axis=1)
    for f in ("fwd", "rev"):
        x = got[f] != want[f]
        int_fail |= x.reshape(n, -1).any(axis=1) & ~badst
    flt_fail = ~close(got["fs_cvg"], want["fs_cvg"], rtol, FS_ATOL) & ~badst
    soft = ((want["flags"] if soft_flags is None else soft_flags) & (capi.FLAG_NEAR_LRT | capi.FLAG_LRT_TIE)) != 0
    call_diff = (got["n_alt"] != want["n_alt"]) | (got["alt"] != want["alt"]).any(axis=1)
    if check_diag:
        call_diff |= got["n_active"] != want["n_active"]
    flips = np.nonzero(call_diff & soft)[0]
    int_fail |= call_diff & ~soft
    same_call = ~call_diff
    for k in range(4):
        live = same_call & (got["n_alt"] > k)
        flt_fail |= live & ~close(got["af"][:, k], want["af"][:, k], rtol)
    flt_fail |= same_call & (got["n_alt"] > 0) & ~close(got["qual"], want["qual"], rtol) & ~soft
    flt_fail |= same_call & (got["n_alt"] > 0) & ~close(got["fs_vcf"], want["fs_vcf"], rtol, FS_ATOL) & ~badst
    if check_diag:
        # sites whose LRT outcome was proven by the bound carry no chi2 (BV_FLAG_LRT_BOUND)
        bound = (got["flags"] & capi.FLAG_LRT_BOUND) != 0
        # chi2 = 2 (LL_full - LL_sub) is a difference of two sums over the site's d reads, which the reference forms read by
        # read: their rounding noise grows with d and does not cancel.  On the 10,000-read rows of BASELINE configs[3] the
        # reference is ~1e-9 away from an 80-bit evaluation of its own formulas, which the histogram sums match to 2e-13
        # (tools/hp_chi2.py, DESIGN.md section 4), so the absolute slack grows with the depth.
        depth = got["depth"].sum(axis=1).astype(np.float64) + got["depth_other"]
        flt_fail |= same_call & ~soft & ~bound & ~close(got["chi2"], want["chi2"], rtol, atol=1e-9 + 1e-12 * depth)
        mask = capi.FLAG_BAD_STRAND
        int_fail |= (got["flags"] & mask) != (want["flags"] & mask)
        int_fail |= same_call & ~soft & ((got["flags"] & capi.FLAG_MONO_QUAL) != (want["flags"] & capi.FLAG_MONO_QUAL))
    return np.nonzero(int_fail)[0], np.nonzero(flt_fail)[0], flips


# ---- the listed flips ----------------------------------------------------------------------------------------------------
# Every parity check that may list flips (a call that differs from the oracle's at a site the ORACLE marks NEAR_LRT / LRT_TIE)
# reports them here under a label.  tests/golden/flips_r02.json holds what the CUDA path produced when the list was last
# regenerated (BV_WRITE_FLIPS=1 writes gpurun_out/flips_observed.json at the end of a GPU run): a check whose label is in the
# file must list exactly those sites -- a kernel change that flips one more call, or one fewer, shows up as a diff of that file.
FLIPS_FILE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "flips_r02.json")
_observed = {}


def committed_flips():
    if not os.path.exists(FLIPS_FILE):
        return {}
    with open(FLIPS_FILE) as f:
        return json.load(f)


def report_flips(label, got, want, flips, soft_flags=None):
    _observed[label] = flip_list(got, want, flips, soft_flags)
    known = committed_flips()
    if label in known and not os.environ.get("BV_WRITE_FLIPS"):
        assert [e["site"] for e in known[label]] == [int(i) for i in flips], \
            f"{label}: flipped sites {[int(i) for i in flips]} differ from the committed list {[e['site'] for e in known[label]]} ({FLIPS_FILE})"


def write_observed_flips(path):
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "w") as f:
        json.dump(_observed, f, indent=1, sort_keys=True)


def flip_list(got, want, flips, soft_flags=None):
    """The listed flips as plain data: site, the oracle's flag, both calls."""
    fl = want["flags"] if soft_flags is None else soft_flags
    return [{"site": int(i), "oracle_flags": int(fl[i]), "cuda_flags": int(got["flags"][i]),
             "cuda_alt": got["alt"][i][:int(got["n_alt"][i])].tolist(), "oracle_alt": want["alt"][i][:int(want["n_alt"][i])].tolist(),
             "cuda_n_active": int(got["n_active"][i]), "oracle_n_active": int(want["n_active"][i])} for i in flips]


def describe(rec):
    return {k: rec[k].tolist() for k in rec.dtype.names}


def random_tile(rng, S, N, cov, qlo, qhi, nalt_max=3, other=0.0, indel=0.0, bad_strand=0.0, pitch=None):
    """Random pileup planes with planted multi-allelic sites, optional junk characters and indels."""
    if pitch is None:
        pitch = (N + 15) // 16 * 16
    base = np.full((S, pitch), 5, np.uint8)
    qual = np.zeros((S, pitch), np.uint8)
    strand = np.full((S, pitch), 2, np.uint8)
    ref = rng.integers(0, 4, S)
    for s in range(S):
        covd = rng.random(N) < cov
        k = rng.integers(0, nalt_max + 1)
        p = np.full(4, 0.002)
        p[ref[s]] = 1.0
        for a in rng.permutation([x for x in range(4) if x != ref[s]])[:k]:
            p[a] = 10 ** rng.uniform(-3, 0)
        p /= p.sum()
        b = rng.choice(4, size=N, p=p).astype(np.uint8)
        u = rng.random(N)
        b[u < other] = 4
        b[(u >= other) & (u < other + indel)] = rng.choice([6, 7])
        base[s, :N] = np.where(covd, b, 5)
        qual[s, :N] = np.where(covd, rng.integers(qlo, qhi + 1, N), 0)
        st = rng.integers(0, 2, N)
        st[rng.random(N) < bad_strand] = 2
        strand[s, :N] = np.where(covd, st, 2)
    refc = np.array([65, 67, 71, 84], np.uint8)[ref]
    return base, qual, strand, refc


N_QBINS = 96   # phred 0..95: the histogram slots of K4a / K6 / K8 that hold one phred each (bv_common.cuh kQSlots)
EM_TASKS = {0: 0, 1: 0, 2: 1, 3: 4, 4: 11}   # EM tasks of a site by its number of active alleles (subsets of >= 2 of them)


def active_threshold(T, min_af):
    """Smallest depth d with (double)d / T >= (double)(float)min_af, the reference's compare (src/basetype.cpp:137)."""
    maf = float(np.float32(min_af))
    d = max(0, int(np.ceil(maf * T)) - 2)
    while d / T < maf:
        d += 1
    return d


def binned_site(rng, nb, k, T, min_af):
    """One row of T counted reads with exactly nb distinct (base, phred) bins (bases A, C, G, T and OTHER, phred 0..95) and
    exactly k active alleles under min_af.  Returns (bases, phreds) in random order, or None when no such row exists.
    Two active alleles always have >= 5 reads each, so that the bound of K3 (REF plus a minor allele of <= 4 reads) never
    settles a site meant for the EM."""
    thr = active_threshold(T, min_af)
    act = np.sort(rng.choice(4, k, replace=False))
    is_act = np.isin(np.arange(5), act)
    cap = np.where(is_act | (np.arange(5) == 4), N_QBINS, min(N_QBINS, thr - 1))
    if k < 1 or nb < k or nb > cap.sum():
        return None
    cnt = is_act.astype(np.int64)
    free = np.repeat(np.arange(5), cap - cnt)
    cnt += np.bincount(rng.choice(free, nb - k, replace=False), minlength=5) if nb > k else 0
    depth = cnt.copy()
    for b in range(4):   # inactive bases: up to one read below the threshold
        if not is_act[b] and cnt[b]:
            depth[b] += rng.integers(0, thr - 1 - cnt[b] + 1)
    if cnt[4]:
        depth[4] += rng.integers(0, max(1, T // 20))
    floor = np.where(is_act, np.maximum(np.maximum(cnt, thr), 5), 0)
    left = T - depth[~is_act].sum() - floor.sum()
    if left < 0:
        depth[~is_act] = cnt[~is_act]
        left = T - depth[~is_act].sum() - floor.sum()
        if left < 0:
            return None
    w = rng.dirichlet(np.ones(k))
    if k >= 2 and rng.random() < 0.3:   # one allele right at the threshold (or at its bin count)
        w[-1] = 0.0
        w /= w.sum()
    depth[act] = floor[act] + rng.multinomial(left, w)
    bases, phreds = [], []
    for b in range(5):
        if depth[b]:
            qs = rng.choice(N_QBINS, cnt[b], replace=False)
            phreds.append(np.concatenate([qs, rng.choice(qs, depth[b] - cnt[b])]))
            bases.append(np.full(depth[b], b))
    order = rng.permutation(T)
    return np.concatenate(bases)[order].astype(np.uint8), np.concatenate(phreds)[order].astype(np.uint8)


def max_bins(k, N, min_af):
    """Most bins binned_tile can place in a row of N cells with k active alleles: 96 per active base and OTHER, and fewer than
    the active threshold of the fewest reads binned_tile covers (90 % of N) per inactive base."""
    return (k + 1) * N_QBINS + (4 - k) * min(N_QBINS, active_threshold(N - N // 10, min_af) - 1)


def deep_shape(rng, S, N, min_af, lo=161):
    """(nb, k) of S deep, wide-phred rows: 1-4 active alleles and more than kSmemBins = 160 bins each (up to max_bins)."""
    ks = [int(k) for k in rng.integers(1, 5, S) if max_bins(int(k), N, min_af) >= lo]
    return [(int(rng.integers(lo, max_bins(k, N, min_af) + 1)), k) for k in ks]


def binned_tile(rng, shape, N, min_af, odd_ref=0.05):
    """Dense planes [S][round16(N)] with one row per (nb, k) of `shape`: exactly nb (base, phred) bins and k active alleles
    (binned_site), 90-100 % of the N cells covered, random strands, REF mostly one of the active alleles, a few 'N' and
    lowercase REFs.  Returns (base, qual, strand, ref_base)."""
    S, pitch = len(shape), (N + 15) // 16 * 16
    base = np.full((S, pitch), 5, np.uint8)
    qual = np.zeros((S, pitch), np.uint8)
    strand = np.full((S, pitch), 2, np.uint8)
    ref = np.zeros(S, np.uint8)
    for s, (nb, k) in enumerate(shape):
        T = N - int(rng.integers(0, N // 10 + 1))
        row = binned_site(rng, nb, k, T, min_af)
        assert row is not None, (nb, k, N, min_af)
        cells = rng.choice(N, T, replace=False)
        base[s, cells], qual[s, cells] = row
        strand[s, cells] = rng.integers(0, 2, T)
        bases = np.unique(row[0][row[0] < 4])
        rc = int(rng.choice(bases)) if len(bases) and rng.random() < 0.7 else int(rng.integers(0, 4))
        u = rng.random()
        ref[s] = ord("N") if u < odd_ref else ord("acgt"[rc]) if u < 2 * odd_ref else ord("ACGT"[rc])
    return base, qual, strand, ref


def bin_counts(base, qual, N):
    """Distinct (base, phred) pairs among the counted cells (base codes 0..4) of every row; phred must be < 96."""
    b, q = base[:, :N].astype(np.int64), qual[:, :N].astype(np.int64)
    counted = b < 5
    assert (q[counted] < N_QBINS).all()
    seen = np.zeros((base.shape[0], 5 * N_QBINS), bool)
    rows = np.broadcast_to(np.arange(base.shape[0])[:, None], b.shape)
    seen[rows[counted], (b * N_QBINS + q)[counted]] = True
    return seen.sum(axis=1)


def active_counts(base, N, min_af):
    """Number of active alleles of every row: depth / total >= min_af (float-widened), total over base codes 0..4."""
    b = base[:, :N]
    depth = np.stack([(b == c).sum(axis=1) for c in range(5)], axis=1)
    total = depth.sum(axis=1)
    with np.errstate(invalid="ignore", divide="ignore"):
        act = (depth[:, :4] / np.maximum(total, 1)[:, None]) >= float(np.float32(min_af))
    return np.where(total > 0, act.sum(axis=1), 0)


def random_aux(rng, base, N, rpr_max=35, mapq_levels=(60, 60, 60, 37, 20, 0)):
    """mapq (u8) and read-position-rank (u16) planes for a base plane; uncovered cells get 0 like the batchfile."""
    S, pitch = base.shape
    mapq = np.zeros((S, pitch), np.uint8)
    rpr = np.zeros((S, (N + 7) // 8 * 8), np.uint16)
    cov = base[:, :N] != 5
    mapq[:, :N] = np.where(cov, rng.choice(np.array(mapq_levels, np.uint8), size=(S, N)), 0)
    rpr[:, :N] = np.where(cov, rng.integers(1, rpr_max + 1, (S, N)), 0)
    return mapq, rpr


def random_groups(rng, N, n_groups, none_frac=0.1):
    g = rng.integers(0, n_groups, N).astype(np.uint8)
    g[rng.random(N) < none_frac] = 255
    return g


def compare_calls(got_calls, got_groups, want_calls, want_groups, rtol=RTOL):
    """Called-site outputs: rank sums bit-exact; group ALT lists exact and AFs within rtol.  Both sorted by site."""
    assert len(got_calls) == len(want_calls), (len(got_calls), len(want_calls))
    bad = []
    for f in ("site", "mq_rank_sum", "read_pos_rank_sum", "base_q_rank_sum"):
        bad += [(f, int(i)) for i in np.nonzero(got_calls[f] != want_calls[f])[0]]
    if want_groups.size:
        assert got_groups.shape == want_groups.shape
        same = (got_groups["n_alt"] == want_groups["n_alt"]) & (got_groups["alt"] == want_groups["alt"]).all(axis=-1)
        bad += [("group_call", tuple(map(int, ix))) for ix in np.argwhere(~same)]
        for k in range(4):
            live = same & (got_groups["n_alt"] > k)
            ok = close(got_groups["af"][..., k], want_groups["af"][..., k], rtol)
            bad += [("group_af", tuple(map(int, ix))) for ix in np.argwhere(live & ~ok)]
    return bad
