"""BAM-driven tile packer and the `basevar basetype` runner (basevar_b200/host/bv_bam, bv_pileup; SURVEY.md 8 rows a17 / f1).

CPU (no GPU needed): our BGZF/BAM/BAI/FASTA readers and the pileup, rendered back into the reference's batchfile text,
against the rows the UNMODIFIED reference command wrote
  * for the committed synthetic BAM fixtures (tests/golden/bam, made by tests/golden/make_golden_bam.py), and
  * for the reference's own bam100 fixture (BASELINE.json configs[0]) when BV_REFERENCE_DIR names its source tree.
GPU: the whole command (BAM -> tiles -> GPU -> VCF / CVG files) against the files the reference command wrote.
"""
import gzip
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tests", "cpp", "bin")
FIX = os.path.join(ROOT, "tests", "golden", "bam")
CLI = os.path.join(ROOT, "basevar_b200", "bin", "basevar")
REF_DIR = os.environ.get("BV_REFERENCE_DIR")   # the original BaseVar source tree, for the test over its own bam100 fixture
REF_DATA = os.path.join(REF_DIR, "tests", "data", "140k_thalassemia_brca_bam") if REF_DIR else ""
N_SAMPLES = 12


@pytest.fixture(scope="module")
def host_built(built_lib):
    from basevar_b200 import build
    build.build_host()
    return BIN


@pytest.fixture(scope="module")
def syn(tmp_path_factory):
    """The synthetic fixture unpacked: plain FASTA (the readers take no compressed FASTA) and a BAM list."""
    d = tmp_path_factory.mktemp("synbam")
    with gzip.open(os.path.join(FIX, "ref.fa.gz"), "rb") as fi, open(d / "ref.fa", "wb") as fo:
        shutil.copyfileobj(fi, fo)
    with open(d / "bam.list", "w") as f:
        for i in range(N_SAMPLES):
            f.write(os.path.join(FIX, "s%02d.bam" % i) + "\n")
    return d


def _dump(host_built, fasta, bamlist, region, *extra):
    p = subprocess.run([os.path.join(host_built, "pileup_dump"), str(fasta), str(bamlist), region, "10", "4", *map(str, extra)],
                       capture_output=True, timeout=900)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    return p.stdout


def _covered(rows):
    return [l for l in rows.split(b"\n") if l and not l.startswith(b"#") and l.split(b"\t", 4)[3] != b"0"]


def test_packer_matches_reference_batchfile_rows_on_synthetic_bams(host_built, syn):
    want = gzip.open(os.path.join(FIX, "rows.covered.txt.gz"), "rb").read()
    want_hdr = [l for l in want.split(b"\n") if l.startswith(b"#")][:3]
    want_rows = [l for l in want.split(b"\n") if l and not l.startswith(b"#")]
    a = _dump(host_built, syn / "ref.fa", syn / "bam.list", "ctgA:1-4000")
    b = _dump(host_built, syn / "ref.fa", syn / "bam.list", "ctgB:10001-520000")
    assert a.split(b"\n")[:3] == want_hdr          # format line, ##SampleIDs= from the first @RG's SM, column names
    assert a.count(b"\n") == 3 + 4000 and b.count(b"\n") == 3 + 510000   # one row per position, covered or not
    got = _covered(a) + _covered(b)
    assert len(got) == len(want_rows) == 7244
    assert got == want_rows
    # the fixture does hold what it was built to hold
    assert sum(l.split(b"\t")[5].count(b"+") for l in want_rows) > 100      # insertions that won a position
    assert any(b" -" in l.split(b"\t")[5] or l.split(b"\t")[5].startswith(b"-") for l in want_rows)   # a deletion that did


@pytest.mark.parametrize("span,tile", [(1000, 64), (4096, 1000), (77777, 333)])
def test_packer_is_independent_of_span_and_tile_sizes(host_built, syn, span, tile):
    """Positions decoded per pass and rows per tile are ours to choose: the reference's 500-kb step survives only as the
    rule for indels anchored on a step's last position (ctgB:510000 in the fixture)."""
    base = _dump(host_built, syn / "ref.fa", syn / "bam.list", "ctgB:10001-520000")
    assert _dump(host_built, syn / "ref.fa", syn / "bam.list", "ctgB:10001-520000", span, tile) == base


def test_index_queries_match_a_linear_scan(host_built):
    for i in (0, 5, 10, 11):
        p = subprocess.run([os.path.join(host_built, "pileup_dump"), "--query-check", os.path.join(FIX, "s%02d.bam" % i), str(i + 1), "400"],
                           capture_output=True, text=True, timeout=300)
        assert p.returncode == 0 and "query-check ok" in p.stdout, p.stdout + p.stderr


def test_bgzf_writer_round_trip(host_built, tmp_path):
    for n in (0, 1, 65280, 65281, 1000003):
        out = tmp_path / ("rt%d.txt.gz" % n)
        p = subprocess.run([os.path.join(host_built, "pileup_dump"), "--bgzf-roundtrip", str(out), str(n), "7"], capture_output=True, text=True, timeout=300)
        assert p.returncode == 0 and "bgzf-roundtrip ok" in p.stdout, p.stdout + p.stderr
        assert len(gzip.open(out, "rb").read()) == n                 # a series of gzip members, as bgzip writes
        assert open(out, "rb").read()[-28:] == bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")   # BGZF EOF marker


def test_unknown_contig_fails_like_the_reference(host_built, syn):
    p = subprocess.run([os.path.join(host_built, "pileup_dump"), str(syn / "ref.fa"), str(syn / "bam.list"), "ctgA:1-10", "10", "2"],
                       capture_output=True, text=True, timeout=300)
    assert p.returncode == 0
    fa = syn / "other.fa"
    fa.write_text(">ctgZ\nACGTACGTAC\n")
    p = subprocess.run([os.path.join(host_built, "pileup_dump"), str(fa), str(syn / "bam.list"), "ctgZ:1-10", "10", "2"],
                       capture_output=True, text=True, timeout=300)
    assert p.returncode != 0 and "Fail to fetch the alignment data" in p.stderr   # src/bam.cpp:93-98


@pytest.mark.skipif(not os.path.isdir(REF_DATA), reason="needs the reference's bam100 fixture: set BV_REFERENCE_DIR to its source tree")
def test_packer_matches_reference_batchfiles_on_bam100(host_built, tmp_path_factory):
    """BASELINE.json configs[0]: the 100 BAM files of the reference's own test, over both regions of its work.log.sh;
    every row equals the batchfile the unmodified reference wrote (tests/golden/c1: of chr17 the rows it keeps)."""
    from tests.golden import make_golden_cli as G
    work = str(tmp_path_factory.mktemp("bam100"))
    bams = [os.path.join(REF_DATA, l.strip()) for l in open(os.path.join(REF_DATA, "bam100.list")) if l.strip()]
    fa = os.path.join(work, "standin.fa")
    G.build_fasta(bams, fa)
    lst = os.path.join(work, "bam.list")
    with open(lst, "w") as f:
        f.write("\n".join(bams) + "\n")
    for region, fn in (("chr11:5246595-5248428", "batch.chr11_5246595-5248428.1_1.bf.gz"), ("chr17:41197764-41276135", G.SAMPLED_BF)):
        want = gzip.open(os.path.join(ROOT, "tests", "golden", "c1", fn), "rb").read().split(b"\n")
        got = _dump(host_built, fa, lst, region).split(b"\n")
        beg, end = map(int, region.split(":")[1].split("-"))
        assert got[:3] == want[:3] and len(got) == 3 + end - beg + 1 + 1   # header, one row per position
        kept = {l.split(b"\t", 2)[1] for l in want[3:] if l}
        assert [l for l in got[3:] if l and l.split(b"\t", 2)[1] in kept] == [l for l in want[3:] if l]


RANGE = os.path.join(ROOT, "tests", "golden", "range")


def test_bgzf_fasta_and_the_references_own_tiny_fixture(host_built, tmp_path):
    """/root/reference/tests/data/work.log.sh:1 -- `-R ce.fa.gz -I range.bam -I range.bam`: a bgzip-compressed FASTA with no
    .fai beside it (src/fasta.cpp:9-48 -> fai_load builds the index), one sample.  Our rows == the batchfile rows the
    unmodified reference wrote for it (tests/golden/make_golden_range.py)."""
    lst = tmp_path / "bam.list"
    lst.write_text(os.path.join(RANGE, "range.bam") + "\n")
    want = gzip.open(os.path.join(RANGE, "batch.rows.txt.gz"), "rb").read()
    got = _dump(host_built, os.path.join(RANGE, "ce.fa.gz"), lst, "CHROMOSOME_I:900-1200")
    assert got == want and got.count(b"\n") == 3 + 301
    # the same text from the plain FASTA and from a compressed one that has its .fai
    with gzip.open(os.path.join(RANGE, "ce.fa.gz"), "rb") as fi, open(tmp_path / "ce.fa", "wb") as fo:
        shutil.copyfileobj(fi, fo)
    assert _dump(host_built, tmp_path / "ce.fa", lst, "CHROMOSOME_I:900-1200") == want
    # plain gzip is refused, as by faidx
    with open(tmp_path / "plain.fa.gz", "wb") as fo:
        fo.write(gzip.compress(b">c\nACGT\n"))
    p = subprocess.run([os.path.join(host_built, "pileup_dump"), str(tmp_path / "plain.fa.gz"), str(lst), "c:1-4", "10", "1"], capture_output=True, text=True)
    assert p.returncode != 0 and "bgzip" in p.stderr


def test_csi_index(host_built, tmp_path):
    """A BAM file with a CSI index only (written by the reference's htslib, min_shift 14): same rows, and index queries
    equal a linear scan."""
    bam = tmp_path / "range_csi.bam"
    shutil.copy(os.path.join(RANGE, "range.bam"), bam)
    shutil.copy(os.path.join(RANGE, "range_csi.bam.csi"), str(bam) + ".csi")
    lst = tmp_path / "bam.list"
    lst.write_text(str(bam) + "\n")
    want = gzip.open(os.path.join(RANGE, "batch.rows.txt.gz"), "rb").read()
    assert _dump(host_built, os.path.join(RANGE, "ce.fa.gz"), lst, "CHROMOSOME_I:900-1200") == want
    p = subprocess.run([os.path.join(host_built, "pileup_dump"), "--query-check", str(bam), "3", "300"], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0 and "query-check ok" in p.stdout, p.stdout + p.stderr


def _rows(text):
    return [l for l in text.split("\n") if l and not l.startswith("##")]


def _meta(text):
    """'##' header lines without the ones that carry file paths (contig assembly=, reference=)."""
    return [l for l in text.split("\n") if l.startswith("##") and not l.startswith("##contig=") and not l.startswith("##reference=")]


@pytest.mark.gpu
@pytest.mark.parametrize("tag,tile,gz,dense", [("syn", 8192, False, False), ("syng", 1000, True, False), ("syn", 129, False, False),
                                               ("syng", 8192, False, True), ("syn", 1000, False, True)])
def test_command_end_to_end_on_synthetic_bams_gpu(host_built, syn, tmp_path, tag, tile, gz, dense):
    """`basevar basetype` over BAM files, no batchfiles: VCF and CVG equal what the unmodified reference command wrote
    (header lines apart from the two that hold file paths, and every row, byte for byte)."""
    vcf = tmp_path / ("out.vcf" + (".gz" if gz else ""))
    cvg = tmp_path / ("out.cvg" + (".gz" if gz else ""))
    cmd = [CLI, "basetype", "-R", str(syn / "ref.fa"), "-L", str(syn / "bam.list"), "-r", "ctgA,ctgB:10001-520000", "-q", "10", "-B", "200",
           "-t", "4", "--output-vcf", str(vcf), "--output-cvg", str(cvg), "--tile-sites", str(tile)]
    if tag == "syng":
        cmd += ["-G", os.path.join(FIX, "groups.info")]
    if dense:   # the packed planes cross PCIe instead of the covered cells (the default): same text either way
        cmd += ["--dense-upload"]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    rd = (lambda f: gzip.open(f, "rt").read()) if gz else (lambda f: open(f).read())
    got_v, got_c = rd(vcf), rd(cvg)
    want_v = gzip.open(os.path.join(FIX, tag + ".vcf.gz"), "rt").read()
    want_c = gzip.open(os.path.join(FIX, tag + ".cvg.gz"), "rt").read()
    assert _meta(got_v) == _meta(want_v)
    assert sum(l.startswith("##contig=") for l in got_v.split("\n")) == 2
    assert _rows(got_v) == _rows(want_v) and len(_rows(want_v)) == 1 + 29
    assert got_c == want_c


@pytest.mark.gpu
def test_command_on_the_references_own_tiny_fixture_gpu(host_built, tmp_path):
    """The reference's own end-to-end test command (tests/data/work.log.sh:1), options spelled as there: VCF rows at 962, 1006,
    1028, 1035, 1045 with QUAL 0.000000 LowQual CM_DP=2 (SURVEY.md 8c), CVG text identical."""
    vcf, cvg = tmp_path / "vz.vcf", tmp_path / "t.cvg"
    bam = os.path.join(RANGE, "range.bam")
    cmd = [CLI, "basetype", "--mapq=10", "--min-af=0.05", "--batch-count=1", "--thread=1", "--regions=CHROMOSOME_I:900-1200",
           "--output-vcf", str(vcf), "--output-cvg", str(cvg), "-R", os.path.join(RANGE, "ce.fa.gz"), "-I", bam, "-I", bam]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    want_v = gzip.open(os.path.join(RANGE, "vz.vcf.gz"), "rt").read()
    want_c = gzip.open(os.path.join(RANGE, "t.cvg.gz"), "rt").read()
    got_v, got_c = open(vcf).read(), open(cvg).read()
    assert _meta(got_v) == _meta(want_v)
    assert _rows(got_v) == _rows(want_v) and [l.split("\t")[1] for l in _rows(got_v)[1:]] == ["962", "1006", "1028", "1035", "1045"]
    assert got_c == want_c


def _gpu_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.gpu
def test_command_sharded_over_several_gpus(host_built, syn, tmp_path):
    """`--gpus 0,1,...`: one host worker and one context per GPU, contiguous region shards cut at the reference's 100-kb task
    boundaries, texts merged in coordinate order (shards that are not next in line spill to temporary files): the files equal
    those of a single-GPU run byte for byte.  Needs >= 2 GPUs (the driver's multi-GPU box, `gpurun --gpus N`)."""
    n = _gpu_count()
    if n < 2:
        pytest.skip("one GPU visible")
    outs = {}
    for tag, gpus in (("one", "0"), ("all", ",".join(str(i) for i in range(min(n, 8))))):
        vcf, cvg = tmp_path / (tag + ".vcf"), tmp_path / (tag + ".cvg")
        cmd = [CLI, "basetype", "-R", str(syn / "ref.fa"), "-L", str(syn / "bam.list"), "-r", "ctgA,ctgB:10001-520000", "-q", "10", "-B", "200",
               "-t", "8", "--output-vcf", str(vcf), "--output-cvg", str(cvg), "--tile-sites", "1000", "--gpus", gpus,
               "-G", os.path.join(FIX, "groups.info")]
        p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
        assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
        outs[tag] = (open(vcf).read(), open(cvg).read())
        assert not [f for f in os.listdir(tmp_path) if f.endswith(".tmp")]   # spill files are gone
    assert outs["one"] == outs["all"]
    want_c = gzip.open(os.path.join(FIX, "syng.cvg.gz"), "rt").read()
    assert outs["all"][1] == want_c
