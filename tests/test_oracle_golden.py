"""CPU tests (no GPU): the oracle restatement + the repository's host code against outputs of the UNMODIFIED reference.

test_oracle_cli_matches_golden   committed goldens (tests/golden/tiny.tar.gz, produced by oracle/_ref/STAR; see make_golden.py)
test_oracle_vs_live_reference    fresh seeded reads through the oracle vs outputs of oracle/_ref/STAR (refcmp.json; see make_golden_refcmp.py)
"""
import os
import subprocess

import pytest

import conftest as cf
import oracle_capi as oc

ROOT = cf.ROOT


def _run_cli(binary, genome_dir, files, out, extra=(), threads=2, env=None):
    cmd = [binary, "--genomeDir", genome_dir, "--readFilesIn"] + files + ["--outFileNamePrefix", out, "--runThreadN", str(threads)] + list(extra)
    subprocess.check_call(cmd, stdout=subprocess.DEVNULL, env=env)


def _opts():
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(ROOT, "tests", "golden", "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    return mg.OPTS


@pytest.mark.parametrize("name", ["std", "hard", "se", "std_opts"])
def test_oracle_cli_matches_golden(oracle, golden, tmp_path, name):
    base = "std" if name == "std_opts" else name
    files = [os.path.join(golden, base + "_1.fq")] + ([os.path.join(golden, base + "_2.fq")] if base != "se" else [])
    out = str(tmp_path) + "/"
    _run_cli(oc.ORACLE_CLI, os.path.join(golden, "idx"), files, out, extra=_opts() if name == "std_opts" else ())
    ref = os.path.join(golden, "ref_" + name)
    assert cf.sam_body(out + "Aligned.out.sam") == cf.sam_body(os.path.join(ref, "Aligned.out.sam"))
    assert open(out + "SJ.out.tab", "rb").read() == open(os.path.join(ref, "SJ.out.tab"), "rb").read()
    assert cf.log_counters(out + "Log.final.out") == cf.log_counters(os.path.join(ref, "Log.final.out"))


def test_sam_header_sq_lines(oracle, golden, tmp_path):
    out = str(tmp_path) + "/"
    _run_cli(oc.ORACLE_CLI, os.path.join(golden, "idx"), [os.path.join(golden, "se_1.fq")], out)
    ours = [l for l in open(out + "Aligned.out.sam") if l.startswith("@HD") or l.startswith("@SQ")]
    ref = [l for l in open(os.path.join(golden, "ref_se", "Aligned.out.sam")) if l.startswith("@HD") or l.startswith("@SQ")]
    assert ours == ref


LIVE_READS = [dict(n_pairs=3000, read_len=100, mm=0.01, seed=77, indel=0.002, nrate=0.002, junk=0.02),
              dict(n_pairs=800, read_len=125, mm=0.04, seed=78, indel=0.003, nrate=0.003, junk=0.0)]
OPTION_SETS = [
    ("hard", ["--outFilterMismatchNoverLmax", "0.1", "--scoreGenomicLengthLog2scale", "0", "--alignSJoverhangMin", "8"]),
    ("std", ["--outSAMattributes", "NH", "HI", "AS", "nM", "XS"]),                      # XS implies --outSAMstrandField intronMotif (Parameters_samAttributes.cpp:172-179)
    ("std", ["--outSAMstrandField", "intronMotif", "--outFilterIntronMotifs", "RemoveNoncanonical"]),
    ("std", ["--alignEndsType", "Extend5pOfRead1", "--outSAMprimaryFlag", "AllBestScore"]),
    ("std", ["--outFilterMultimapNmax", "3", "--winAnchorMultimapNmax", "100", "--outSAMmultNmax", "2"]),
]


@pytest.mark.parametrize("kw", LIVE_READS)
def test_oracle_vs_live_reference(oracle, golden, refcmp, tmp_path, kw):
    """Fresh seeded reads (not in tiny.tar.gz): oracle vs the unmodified reference binary (refcmp.json), byte-identical outputs."""
    import hashlib
    import synth
    ref = refcmp("live", kw)
    chrs = synth.make_genome("tiny")
    trs = synth.make_annotation(chrs, "tiny")
    m1, m2 = synth.make_reads(chrs, trs, **kw)
    f1, f2 = str(tmp_path / "r_1.fq"), str(tmp_path / "r_2.fq")
    synth.write_fastq(m1, f1)
    synth.write_fastq(m2, f2)
    assert [hashlib.sha256(open(f, "rb").read()).hexdigest() for f in (f1, f2)] == ref["reads_sha256"], \
        "tools/synth.py no longer makes the reads the reference outputs belong to"
    _run_cli(oc.ORACLE_CLI, os.path.join(golden, "idx"), [f1, f2], str(tmp_path) + "/", threads=2)
    assert cf.run_summary(str(tmp_path) + "/") == ref["outputs"]


@pytest.mark.parametrize("base,extra", OPTION_SETS)
def test_option_sets_vs_live_reference(oracle, golden, refcmp, tmp_path, base, extra):
    """Non-default option sets that are not in tiny.tar.gz: oracle-driven host code vs the unmodified reference binary (refcmp.json)."""
    files = [os.path.join(golden, base + "_1.fq"), os.path.join(golden, base + "_2.fq")]
    _run_cli(oc.ORACLE_CLI, os.path.join(golden, "idx"), files, str(tmp_path) + "/", extra=extra, threads=2)
    assert cf.run_summary(str(tmp_path) + "/") == refcmp("opts", base, extra)["outputs"]


@pytest.mark.parametrize("name", ["std", "hard", "se"])
def test_kary_seed_search_design_check(oracle, lib, golden, name, monkeypatch):
    """Design check for the next GPU seed-search kernel: a 32-ary search (the shape a warp executes cooperatively) must return the
    same maximal match length and the same block of SA rows as the reference's binary search (SuffixArrayFuns.cpp:133-207) for every
    search of the read set — emulated lane by lane inside the oracle (oracle/star_oracle.cpp, karyMaxMappableLength)."""
    import ctypes as C
    import star_b200 as sb
    monkeypatch.setenv("STAR_ORACLE_KARY_CHECK", "1")
    files = [os.path.join(golden, name + "_1.fq")] + ([os.path.join(golden, name + "_2.fq")] if name != "se" else [])
    mates = [cf.read_fastq_seqs(f) for f in files]
    seq, off, n, nm = sb.pack_reads(mates)
    idx = sb.Index(lib, os.path.join(golden, "idx"))
    oracle.star_oracle_kary_stats.argtypes = [C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    a0, b0 = C.c_uint64(), C.c_uint64()
    oracle.star_oracle_kary_stats(C.byref(a0), C.byref(b0))
    oe = oc.OracleEngine(oracle, idx)
    oe.map_chunk(seq, off, n, nm)
    oe.close()
    idx.close()
    a1, b1 = C.c_uint64(), C.c_uint64()
    oracle.star_oracle_kary_stats(C.byref(a1), C.byref(b1))
    assert a1.value - a0.value > 1000, "the check did not run"
    assert b1.value - b0.value == 0
