"""The bit-identity gate of BASELINE.json configs[0] at its real size, on the GPU (SURVEY.md §8(c), last bullet).

Genome: the chr21-sized synthetic stand-in (46.7 Mb, 3 chromosomes, repeat families, N block, 1352 spliced transcripts -> sjdb; there is no
real chr21 on the box), index built on the box by this repository's GPU genomeGenerate, whose files must equal the UNMODIFIED reference's
(SHA-256 digests in tests/golden/gate_chr21.json, see make_golden_gate.py).  The drop-in command line star_b200/bin/STAR (CUDA engine) maps
seeded FASTQ files; the SAM records, SJ.out.tab and the integer counters of Log.final.out must equal those of oracle/_ref/STAR
--runThreadN 1 on the same files (record count + digests, counters as text, in the same JSON file):
  * 100 k pairs 2x100 at 0.5 % substitutions (configs[0]),
  * 20 k pairs 2x150 at 5 % substitutions (configs[2] shape: long recursion trees, pool / task caps, overflow tiers),
and the engine's records for the same reads equal the oracle's field by field through the C-ABI.  The heavy tail that drives the
design (windows with 35-45 seeds from the repeat families, tens of thousands of recursion nodes per read, bump pools with per-chunk
offsets) only exists at this size.  Also here: both suffix-sort paths of the GPU genomeGenerate reproduce the reference's index files.
"""
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

import conftest as cf

pytestmark = pytest.mark.gpu

ROOT = cf.ROOT
OURS = os.path.join(ROOT, "star_b200", "bin", "STAR")
GOLDEN = os.path.join(ROOT, "tests", "golden", "gate_chr21.json")
CASES = [("std100", 100_000, 100, 0.005), ("hard150", 20_000, 150, 0.05)]
INDEX_FILES = ("Genome", "SA", "SAindex", "chrStart.txt", "chrLength.txt", "chrName.txt", "sjdbInfo.txt", "sjdbList.out.tab", "exonInfo.tab",
               "transcriptInfo.tab")


@pytest.fixture(scope="module")
def chr21(tmp_path_factory):
    """Work directory with genome.fa, annot.gtf and idx/ (this repository's genomeGenerate); shared with bench.py --preset chr21."""
    import bench
    import synth
    wd = os.path.join(os.environ.get("STAR_B200_BENCH_DIR", "/tmp/star_b200_bench"), "chr21")
    os.makedirs(wd, exist_ok=True)
    chrs, trs, idx, _ = bench.prepare_genome(wd, "chr21", own_generate=True)
    with open(GOLDEN) as f:
        golden = json.load(f)
    return {"dir": wd, "chrs": chrs, "trs": trs, "idx": idx, "synth": synth, "golden": golden}


def digest(p):
    h = hashlib.sha256()
    with open(p, "rb") as f:
        for blk in iter(lambda: f.read(1 << 24), b""):
            h.update(blk)
    return h.hexdigest()


def _reads(c, n, read_len, mm, seed, tag):
    s = c["synth"]
    m1, m2 = s.make_reads(c["chrs"], c["trs"], n, read_len=read_len, mm=mm, seed=seed)
    f1, f2 = os.path.join(c["dir"], tag + "_1.fq"), os.path.join(c["dir"], tag + "_2.fq")
    s.write_fastq(m1, f1)
    s.write_fastq(m2, f2)
    return m1, m2, f1, f2


def _run(binary, idx, f1, f2, out, extra=()):
    os.makedirs(out, exist_ok=True)
    subprocess.check_call([binary, "--genomeDir", idx, "--readFilesIn", f1, f2, "--outFileNamePrefix", out + "/"] + list(extra), stdout=subprocess.DEVNULL, timeout=1500)


@pytest.mark.parametrize("name,n,read_len,mm", CASES)
def test_cli_equals_reference_at_config_size(lib, chr21, tmp_path, name, n, read_len, mm):
    for f in INDEX_FILES:   # the outputs below are the reference's on its own index
        assert digest(os.path.join(chr21["idx"], f)) == chr21["golden"]["index_sha256"][f], f
    ref = chr21["golden"]["cases"][name]
    _, _, f1, f2 = _reads(chr21, n, read_len, mm, 77, "gate_" + name)
    assert [digest(f) for f in (f1, f2)] == ref["reads_sha256"], "tools/synth.py no longer makes the reads the reference outputs belong to"
    ours = str(tmp_path / "ours")
    _run(OURS, chr21["idx"], f1, f2, ours, ["--runThreadN", "16"])
    assert cf.run_summary(ours + "/") == ref["outputs"]


@pytest.mark.parametrize("name,n,read_len,mm", CASES)
def test_engine_equals_oracle_at_config_size(lib, oracle, chr21, name, n, read_len, mm):
    """Through the C-ABI, one chunk: every field of every record, plus the work counters the roofline numerator is built from."""
    import oracle_capi as oc
    import star_b200 as sb
    m1, m2, _, _ = _reads(chr21, n, read_len, mm, 78, "gate2_" + name)
    seq, off, n_, nm = sb.pack_reads([m1, m2])
    index = sb.Index(lib, chr21["idx"])
    try:
        eng = sb.Engine(lib, index, max_reads=n_)
        res_g, al_g, st_g = eng.map_chunk(seq, off, n_, nm)
        eng.close()
        oe = oc.OracleEngine(oracle, index)
        res_o, al_o, st_o = oe.map_chunk(seq, off, n_, nm)
        oe.close()
    finally:
        index.close()
    diffs = oc.compare_outputs(res_o, al_o, res_g, al_g)
    assert not diffs, "\n".join(diffs[:20])
    for k in ("mmp_searches", "mmp_sai_words", "sa_enumerated"):
        assert getattr(st_g, k) == getattr(st_o, k), k


def test_gpu_generate_equals_reference_index_at_config_size(lib, chr21, tmp_path):
    """This repository's --runMode genomeGenerate (GPU suffix sort, both the 32-bit path and the batched 64-bit path that GRCh38 takes)
    writes the reference's Genome / SA / SAindex / junction files for the chr21-sized genome byte for byte."""
    ref = chr21["golden"]["index_sha256"]
    for tag, env in (("small_path", {}), ("large_path", {"STAR_B200_SA_LARGE_CAP": "30000000"})):
        out = str(tmp_path / tag)
        os.makedirs(out)
        subprocess.check_call([OURS, "--runMode", "genomeGenerate", "--genomeDir", out, "--genomeFastaFiles", os.path.join(chr21["dir"], "genome.fa"),
                               "--sjdbGTFfile", os.path.join(chr21["dir"], "annot.gtf"), "--sjdbOverhang", "99", "--genomeSAindexNbases", "11", "--runThreadN", "16",
                               "--outFileNamePrefix", out + "_log_"], stdout=subprocess.DEVNULL, env=dict(os.environ, **env), timeout=1500)
        for f in INDEX_FILES:
            assert digest(os.path.join(out, f)) == ref[f], (tag, f)
