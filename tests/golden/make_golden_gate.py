#!/usr/bin/env python3
"""Regenerates tests/golden/gate_chr21.json — run where oracle/_ref/STAR was built (oracle/Makefile.ref).

What tests/test_gpu_config_gate.py compares against, from the UNMODIFIED reference binary on the chr21-sized synthetic genome
(tools/synth.py preset chr21, built by bench.prepare_genome, i.e. the reference's --runMode genomeGenerate):

  index_sha256   SHA-256 of the index files the reference wrote (test_gpu_config_gate.INDEX_FILES)
  cases/<name>   for each of test_gpu_config_gate.CASES: reads_sha256 (the two FASTQ files, seed 77) and the summary of the reference's
                 outputs with --runThreadN 1 (conftest.run_summary: SAM record count + digest, SJ.out.tab digest, Log.final.out counters)

The outputs themselves (an index of ~0.5 GB, SAM files of tens of MB) are too large to commit.
"""
import json
import os
import shutil
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
import conftest as cf  # noqa: E402
import synth  # noqa: E402
import test_gpu_config_gate as gate  # noqa: E402


def main():
    assert os.path.exists(bench.REF_STAR), "build oracle/_ref/STAR first (make -f oracle/Makefile.ref)"
    os.environ.pop("STAR_B200_BENCH_OWN_GENERATE", None)
    tmp = tempfile.mkdtemp(prefix="golden_gate_")
    chrs, trs, idx, info = bench.prepare_genome(tmp, "chr21")
    assert info["builder"].startswith("reference"), info
    table = {"index_sha256": {f: gate.digest(os.path.join(idx, f)) for f in gate.INDEX_FILES}, "cases": {}}
    c = {"dir": tmp, "chrs": chrs, "trs": trs, "synth": synth}
    for name, n, read_len, mm in gate.CASES:
        _, _, f1, f2 = gate._reads(c, n, read_len, mm, 77, "gate_" + name)
        out = os.path.join(tmp, "ref_" + name)
        gate._run(bench.REF_STAR, idx, f1, f2, out, ["--runThreadN", "1"])
        table["cases"][name] = {"reads_sha256": [gate.digest(f) for f in (f1, f2)], "outputs": cf.run_summary(out + "/")}
        print(name, table["cases"][name]["outputs"]["sam_records"], "records", file=sys.stderr)
    dst = os.path.join(ROOT, "tests", "golden", "gate_chr21.json")
    with open(dst, "w") as f:
        json.dump(table, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", dst, os.path.getsize(dst), "bytes")
    shutil.rmtree(tmp)


if __name__ == "__main__":
    main()
