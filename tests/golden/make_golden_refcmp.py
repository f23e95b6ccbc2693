#!/usr/bin/env python3
"""Regenerates tests/golden/refcmp.json — run where oracle/_ref/STAR was built (oracle/Makefile.ref).

Outputs of the UNMODIFIED reference binary for the comparisons that are not in tiny.tar.gz, on the inputs of tiny.tar.gz and with
the command lines the tests use (the case lists are imported from the test modules).  The outputs themselves are too large to
commit, so each case keeps what its test compares, reduced to counts and SHA-256 digests (conftest.run_summary,
test_bam_output.bam_summary); the Log.final.out counters, BAM header lines and @RG lines are kept as text:

  live    fresh seeded reads (test_oracle_golden.LIVE_READS; tools/synth.py makes them again at test time, reads_sha256 pins them)
  opts    non-default option sets on the std / hard reads (test_oracle_golden.OPTION_SETS)
  bam     --outSAMtype BAM Unsorted (test_bam_output.CASES), reference --runThreadN 1
  sorted  --outSAMtype BAM Unsorted SortedByCoordinate (test_bam_output.SORT_CASES), reference --runThreadN 2: the sorted file, and
          the unsorted one as a multiset of records (its order depends on the reference's threads)
  rg      comma-separated file lists with one read group per file (test_host_pipeline.RG_MODES)

Key of a case: conftest.refcmp_key(group, parameters).
"""
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tarfile
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import conftest as cf  # noqa: E402
import synth  # noqa: E402
import test_bam_output as tbo  # noqa: E402
import test_host_pipeline as thp  # noqa: E402
import test_oracle_golden as tog  # noqa: E402

STAR = os.path.join(ROOT, "oracle", "_ref", "STAR")


def run(cmd, out):
    os.makedirs(out)
    subprocess.check_call(cmd, cwd=out, stdout=subprocess.DEVNULL)
    return out + "/"


def main():
    tmp = tempfile.mkdtemp(prefix="golden_refcmp_")
    with tarfile.open(os.path.join(ROOT, "tests", "golden", "tiny.tar.gz")) as t:
        t.extractall(tmp)
    g = os.path.join(tmp, "tiny")
    idx = os.path.join(g, "idx")
    table = {}

    def case(group, *params):
        return os.path.join(tmp, "runs", "%s_%d" % (group, len(table))), cf.refcmp_key(group, *params)

    chrs = synth.make_genome("tiny")
    trs = synth.make_annotation(chrs, "tiny")
    for kw in tog.LIVE_READS:
        d, k = case("live", kw)
        m1, m2 = synth.make_reads(chrs, trs, **kw)
        f1, f2 = os.path.join(tmp, "r_1.fq"), os.path.join(tmp, "r_2.fq")
        synth.write_fastq(m1, f1)
        synth.write_fastq(m2, f2)
        out = run([STAR, "--genomeDir", idx, "--readFilesIn", f1, f2, "--outFileNamePrefix", d + "/", "--runThreadN", "1"], d)
        table[k] = {"reads_sha256": [hashlib.sha256(open(f, "rb").read()).hexdigest() for f in (f1, f2)], "outputs": cf.run_summary(out)}
    for base, extra in tog.OPTION_SETS:
        d, k = case("opts", base, extra)
        files = [os.path.join(g, base + "_1.fq"), os.path.join(g, base + "_2.fq")]
        out = run([STAR, "--genomeDir", idx, "--readFilesIn"] + files + ["--outFileNamePrefix", d + "/", "--runThreadN", "1"] + extra, d)
        table[k] = {"outputs": cf.run_summary(out)}
    for base, extra in tbo.CASES:
        d, k = case("bam", base, extra)
        out = run([STAR, "--genomeDir", idx, "--readFilesIn"] + tbo.input_files(g, base) + ["--outFileNamePrefix", d + "/", "--runThreadN", "1",
                   "--outSAMtype", "BAM", "Unsorted"] + extra, d)
        table[k] = {"bam": tbo.bam_summary(*tbo.parse_bam(out + "Aligned.out.bam")[1:])}
    for base, extra in tbo.SORT_CASES:
        d, k = case("sorted", base, extra)
        out = run([STAR, "--genomeDir", idx, "--readFilesIn"] + tbo.input_files(g, base) + ["--outFileNamePrefix", d + "/", "--runThreadN", "2",
                   "--outSAMtype", "BAM", "Unsorted", "SortedByCoordinate"] + extra, d)
        _, text, refs, recs = tbo.parse_bam(out + "Aligned.out.bam")
        table[k] = {"sorted": tbo.bam_summary(*tbo.parse_bam(out + "Aligned.sortedByCoord.out.bam")[1:]),
                    "unsorted_as_multiset": tbo.bam_summary(text, refs, sorted(recs))}
    for mode in thp.RG_MODES:
        d, k = case("rg", mode)
        parts, extra = thp.rg_inputs(g, tmp, mode)
        out = run([STAR, "--genomeDir", idx, "--readFilesIn", parts[1], parts[2], "--outFileNamePrefix", d + "/", "--runThreadN", "1"] + extra, d)
        table[k] = {"outputs": cf.run_summary(out), "rg_header": thp.rg_header_lines(out + "Aligned.out.sam")}
    dst = os.path.join(ROOT, "tests", "golden", "refcmp.json")
    with open(dst, "w") as f:
        json.dump(table, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", dst, os.path.getsize(dst), "bytes,", len(table), "cases")
    shutil.rmtree(tmp)


if __name__ == "__main__":
    main()
