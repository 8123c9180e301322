"""Generate the C1 end-to-end fixtures from the UNMODIFIED reference command line (run HERE only: needs /root/reference).

    bash oracle/build_ref_cli.sh
    gcc -O2 -fPIC -shared -o oracle/_ref/libkeepbf.so oracle/keep_batchfiles.c -ldl
    python tests/golden/make_golden_cli.py

What it does (BASELINE.json configs[0]: `basevar basetype` on the repo's tests/data BAM list, -t 4 -B 200):
  1. builds a stand-in FASTA for the bam100 fixture (the hg19 FASTA the reference's own work.log.sh names is not in the
     repository): every record's CIGAR + MD tag gives the true reference base at each aligned position; all other
     positions are 'N' (SURVEY.md section 8c).  Written to a scratch directory, never committed.
  2. runs oracle/_ref/basevar basetype over the regions of tests/data/140k_thalassemia_brca_bam/work.log.sh:5-8 with
     the batchfiles kept (oracle/keep_batchfiles.c), once with and once without --pop-group;
  3. commits, under tests/golden/c1/: the batchfile rows the reference fed to `_basevar_caller` (gzip text), and the
     VCF / CVG text it wrote for them -- the expected output of our host pipeline on the same rows;
  4. keeps the chr17 batchfile under 1 MB: its called rows and a seeded sample of the others (sample_chr17).
"""
import gzip
import os
import shutil
import struct
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
REF = os.environ.get("BV_REFERENCE_DIR", "/root/reference")
DATA = os.path.join(REF, "tests", "data", "140k_thalassemia_brca_bam")
OUT = os.path.join(ROOT, "tests", "golden", "c1")
BIN = os.path.join(ROOT, "oracle", "_ref", "basevar")
KEEP = os.path.join(ROOT, "oracle", "_ref", "libkeepbf.so")
REGIONS = "chr11:5246595-5248428,chr17:41197764-41276135"
SEQ = "=ACMGRSVTWYHKDBN"


def bam_records(path):
    """(ref_name, pos0, cigar [(op, len)], seq, MD or None) for every mapped record; BGZF is multi-member gzip."""
    with gzip.open(path, "rb") as f:
        data = f.read()
    assert data[:4] == b"BAM\1"
    l_text, = struct.unpack_from("<i", data, 4)
    o = 8 + l_text
    n_ref, = struct.unpack_from("<i", data, o)
    o += 4
    refs = []
    for _ in range(n_ref):
        l_name, = struct.unpack_from("<i", data, o)
        name = data[o + 4:o + 4 + l_name - 1].decode()
        l_ref, = struct.unpack_from("<i", data, o + 4 + l_name)
        refs.append((name, l_ref))
        o += 8 + l_name
    while o < len(data):
        bs, = struct.unpack_from("<i", data, o)
        rec = data[o + 4:o + 4 + bs]
        o += 4 + bs
        ref_id, pos, l_rn, mapq, bin_, n_cig, flag, l_seq = struct.unpack_from("<iiBBHHHi", rec, 0)
        if ref_id < 0 or flag & 4:
            continue
        p = 32 + l_rn
        cigar = [(c & 15, c >> 4) for c in struct.unpack_from("<%dI" % n_cig, rec, p)]
        p += 4 * n_cig
        sq = rec[p:p + (l_seq + 1) // 2]
        seq = "".join(SEQ[(sq[i >> 1] >> (4 * (1 - (i & 1)))) & 15] for i in range(l_seq))
        p += (l_seq + 1) // 2 + l_seq
        md = None
        while p < len(rec):
            tag, typ = rec[p:p + 2], chr(rec[p + 2])
            p += 3
            if typ == "Z" or typ == "H":
                e = rec.index(b"\0", p)
                if tag == b"MD":
                    md = rec[p:e].decode()
                p = e + 1
            elif typ in "AcC":
                p += 1
            elif typ in "sS":
                p += 2
            elif typ in "iIf":
                p += 4
            elif typ == "B":
                sub = chr(rec[p])
                cnt, = struct.unpack_from("<i", rec, p + 1)
                p += 5 + cnt * {"c": 1, "C": 1, "s": 2, "S": 2, "i": 4, "I": 4, "f": 4}[sub]
            else:
                raise ValueError("aux type " + typ)
        yield refs, refs[ref_id][0], pos, cigar, seq, md


def reference_bases(pos, cigar, seq, md):
    """{ref position (0-based): base} from CIGAR + MD."""
    out = {}
    # reference-consuming aligned columns in order, with the read base for M/=/X and None for D
    cols = []
    r, q = pos, 0
    for op, ln in cigar:
        if op in (0, 7, 8):
            for k in range(ln):
                cols.append((r + k, seq[q + k]))
            r += ln
            q += ln
        elif op == 2:
            for k in range(ln):
                cols.append((r + k, None))
            r += ln
        elif op == 3:
            r += ln
        elif op in (1, 4):
            q += ln
    if md is None:
        return out
    i, c = 0, 0
    while i < len(md):
        if md[i].isdigit():
            j = i
            while j < len(md) and md[j].isdigit():
                j += 1
            for _ in range(int(md[i:j])):
                rp, b = cols[c]
                out[rp] = b
                c += 1
            i = j
        elif md[i] == "^":
            i += 1
            while i < len(md) and md[i].isalpha():
                out[cols[c][0]] = md[i]
                c += 1
                i += 1
        else:
            out[cols[c][0]] = md[i]
            c += 1
            i += 1
    return out


def build_fasta(bams, path):
    contigs = {}
    lens = None
    for b in bams:
        for refs, name, pos, cigar, seq, md in bam_records(b):
            if lens is None:
                lens = dict(refs)
            if name not in ("chr11", "chr17"):
                continue
            if name not in contigs:
                contigs[name] = bytearray(b"N" * lens[name])
            arr = contigs[name]
            for rp, base in reference_bases(pos, cigar, seq, md).items():
                if base and 0 <= rp < len(arr):
                    arr[rp] = ord(base.upper())
    with open(path, "wb") as f:
        for name in ("chr11", "chr17"):
            f.write(b">" + name.encode() + b"\n")
            f.write(bytes(contigs.get(name, bytearray(b"N" * lens[name]))))
            f.write(b"\n")


def run(work, tag, extra):
    vcf = os.path.join(work, tag + ".vcf")
    cvg = os.path.join(work, tag + ".cvg")
    lst = os.path.join(work, "bam.list")
    cmd = [BIN, "basetype", "-q", "10", "-B", "200", "-t", "4", "-r", REGIONS, "--output-vcf", vcf, "--output-cvg", cvg,
           "-R", os.path.join(work, "standin.fa"), "-L", lst] + extra
    env = dict(os.environ, LD_PRELOAD=KEEP)
    subprocess.check_call(cmd, env=env, stdout=open(os.path.join(work, tag + ".log"), "w"))
    return vcf, cvg, os.path.join(work, "cache_" + tag)


FULL_BF = "batch.chr17_41197764-41276135.1_1.bf.gz"
SAMPLED_BF = "batch.chr17_41197764-41276135.sampled.bf.gz"


def sample_chr17(out, frac=0.2, seed=17):
    """The chr17 batchfile holds 78,372 rows (3.1 MB compressed); keep every row at a position either VCF calls plus a seeded
    sample `frac` of the others (0.8 MB), and drop the CVG rows of the positions left out.  Every VCF / CVG row comes from its
    own batchfile row, so the reference's text for the kept rows is its text for the whole region, filtered."""
    bf = gzip.open(os.path.join(out, FULL_BF), "rb").read().split(b"\n")
    hdr = [l for l in bf if l.startswith(b"#")]
    rows = [l for l in bf if l and not l.startswith(b"#")]
    called = {int(l.split("\t")[1]) for t in ("c1", "c1g") for l in gzip.open(os.path.join(out, t + ".vcf.gz"), "rt")
              if l.startswith("chr17\t")}
    u = np.random.default_rng(seed).random(len(rows))
    keep = [r for r, x in zip(rows, u) if x < frac or int(r.split(b"\t", 2)[1]) in called]
    kept = {int(r.split(b"\t", 2)[1]) for r in keep}
    with gzip.GzipFile(os.path.join(out, SAMPLED_BF), "wb", mtime=0) as fo:
        fo.write(b"\n".join(hdr + keep) + b"\n")
    for t in ("c1", "c1g"):
        lines = gzip.open(os.path.join(out, t + ".cvg.gz"), "rb").read().split(b"\n")[:-1]
        lines = [l for l in lines if not l.startswith(b"chr17\t") or int(l.split(b"\t", 2)[1]) in kept]
        with gzip.GzipFile(os.path.join(out, t + ".cvg.gz"), "wb", mtime=0) as fo:
            fo.write(b"\n".join(lines) + b"\n")
    os.remove(os.path.join(out, FULL_BF))
    print(f"{SAMPLED_BF}: {len(keep)} of {len(rows)} rows, {len(called)} called positions")


def main():
    work = os.environ.get("BV_GOLDEN_WORK", "/tmp/bv_golden_cli")
    os.makedirs(work, exist_ok=True)
    os.makedirs(OUT, exist_ok=True)
    bams = [os.path.join(DATA, l.strip()) for l in open(os.path.join(DATA, "bam100.list")) if l.strip()]
    with open(os.path.join(work, "bam.list"), "w") as f:
        f.write("\n".join(bams) + "\n")
    fa = os.path.join(work, "standin.fa")
    if not os.path.exists(fa):
        build_fasta(bams, fa)
    for tag, extra in (("c1", []), ("c1g", ["-G", os.path.join(DATA, "sample_group.info")])):
        shutil.rmtree(os.path.join(work, "cache_" + tag), ignore_errors=True)
        vcf, cvg, cache = run(work, tag, extra)
        for src, dst in ((vcf, tag + ".vcf.gz"), (cvg, tag + ".cvg.gz")):
            with open(src, "rb") as fi, gzip.GzipFile(os.path.join(OUT, dst), "wb", mtime=0) as fo:
                fo.write(fi.read())
        if tag == "c1":
            for fn in sorted(os.listdir(cache)):
                if fn.endswith(".tbi") or ".vcf" in fn or ".cvg" in fn:
                    continue
                with gzip.open(os.path.join(cache, fn), "rb") as fi, \
                        gzip.GzipFile(os.path.join(OUT, fn.replace("c1.", "batch.") + ("" if fn.endswith(".gz") else ".gz")), "wb", mtime=0) as fo:
                    fo.write(fi.read())
        print(tag, "done")
    shutil.copy(os.path.join(DATA, "sample_group.info"), os.path.join(OUT, "sample_group.info"))
    sample_chr17(OUT)


if __name__ == "__main__":
    sys.exit(main())
