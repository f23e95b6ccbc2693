import os
import subprocess
import sys
import tarfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu on the GPU box")


@pytest.fixture(scope="session")
def golden(tmp_path_factory):
    """Unpacked tests/golden/tiny.tar.gz (inputs + outputs of the unmodified reference binary)."""
    d = tmp_path_factory.mktemp("golden")
    with tarfile.open(os.path.join(ROOT, "tests", "golden", "tiny.tar.gz")) as t:
        t.extractall(d)
    return str(d / "tiny")


@pytest.fixture(scope="session")
def lib():
    """The product library (built by __graft_entry__.build() / make)."""
    import star_b200
    if not os.path.exists(star_b200.capi.LIB_PATH):
        subprocess.check_call(["make", "-s", "-j8"], cwd=ROOT)
    return star_b200.load_library()


@pytest.fixture(scope="session")
def oracle():
    import oracle_capi
    oracle_capi.build_oracle()
    return oracle_capi.load_oracle()


def read_fastq_seqs(path):
    with open(path, "rb") as f:
        lines = f.read().split(b"\n")
    return lines[1::4]


def sam_body(path):
    with open(path, "rb") as f:
        return [l for l in f.read().split(b"\n") if l and not l.startswith(b"@")]


def log_counters(path):
    """Integer / percentage lines of Log.final.out (times and speed excluded)."""
    out = []
    with open(path) as f:
        for i, l in enumerate(f):
            if "|" not in l:
                continue
            k, v = l.split("|", 1)
            k = k.strip()
            if k.startswith("Started") or k.startswith("Finished") or k.startswith("Mapping speed"):
                continue
            out.append((k, v.strip()))
    return out


@pytest.fixture(scope="session")
def twopass_golden(tmp_path_factory):
    """Unpacked tests/golden/twopass.tar.gz (junction insertion / 2-pass outputs of the unmodified reference; make_golden_twopass.py)."""
    d = tmp_path_factory.mktemp("golden_tp")
    with tarfile.open(os.path.join(ROOT, "tests", "golden", "twopass.tar.gz")) as t:
        t.extractall(d)
    return str(d / "twopass")


def refcmp_key(group, *params):
    """Key of one case in tests/golden/refcmp.json: the group and the case's parameters."""
    import json
    return group + " " + json.dumps(params, sort_keys=True)


@pytest.fixture(scope="session")
def refcmp():
    """tests/golden/refcmp.json: summaries of outputs of the unmodified reference for the cases outside tiny.tar.gz (make_golden_refcmp.py).
    refcmp(group, *params) is the entry of one case."""
    import json
    with open(os.path.join(ROOT, "tests", "golden", "refcmp.json")) as f:
        table = json.load(f)

    def case(group, *params):
        k = refcmp_key(group, *params)
        assert k in table, "no reference outputs for %s: regenerate tests/golden/refcmp.json with tests/golden/make_golden_refcmp.py" % k
        return table[k]
    return case


def sha256_lines(lines):
    import hashlib
    return hashlib.sha256(b"\n".join(lines)).hexdigest()


def run_summary(prefix):
    """Aligned.out.sam (records: count + digest), SJ.out.tab (digest) and the Log.final.out counters of a run, as refcmp.json stores them"""
    import hashlib
    body = sam_body(prefix + "Aligned.out.sam")
    return {"sam_records": len(body), "sam_sha256": sha256_lines(body),
            "sj_out_tab_sha256": hashlib.sha256(open(prefix + "SJ.out.tab", "rb").read()).hexdigest(),
            "log_counters": [list(kv) for kv in log_counters(prefix + "Log.final.out")]}


def check_twopass_outputs(out, ref):
    """Everything the reference writes in a junction-insertion / 2-pass run: records, junctions, counters of both passes, the junction
    database and (by digest) the rebuilt Genome / SA / SAindex."""
    import hashlib
    if os.path.exists(os.path.join(ref, "Aligned.out.sam")):
        assert sam_body(out + "Aligned.out.sam") == sam_body(os.path.join(ref, "Aligned.out.sam"))
    for f in ("Aligned.out.bam", "Aligned.sortedByCoord.out.bam"):   # header lines except @PG ID:STAR / @CO user command line, references, every record
        if os.path.exists(os.path.join(ref, f)):
            import gzip, struct

            def parts(path):
                d = gzip.decompress(open(path, "rb").read())
                lt = struct.unpack("<i", d[4:8])[0]
                text = [l for l in d[8:8 + lt].split(b"\n") if not l.startswith(b"@PG\tID:STAR") and not l.startswith(b"@CO\tuser command line")]
                return text, d[8 + lt:]
            assert parts(out + f) == parts(os.path.join(ref, f)), f
    assert open(out + "SJ.out.tab", "rb").read() == open(os.path.join(ref, "SJ.out.tab"), "rb").read()
    assert log_counters(out + "Log.final.out") == log_counters(os.path.join(ref, "Log.final.out"))
    for f in ("_STARgenome/sjdbInfo.txt", "_STARgenome/sjdbList.out.tab", "_STARgenome/sjdbList.fromGTF.out.tab", "_STARgenome/exonInfo.tab",
              "_STARgenome/transcriptInfo.tab", "_STARgenome/geneInfo.tab", "_STARgenome/exonGeTrInfo.tab", "_STARpass1/SJ.out.tab",
              "Unmapped.out.mate1", "Unmapped.out.mate2", "ReadsPerGene.out.tab"):
        if os.path.exists(os.path.join(ref, f)):
            assert open(out + f, "rb").read() == open(os.path.join(ref, f), "rb").read(), f
    if os.path.exists(os.path.join(ref, "Aligned.toTranscriptome.out.bam")):   # header (@SQ per transcript, @RG), references and every record incl. the drawn primary flags
        import gzip
        assert gzip.decompress(open(out + "Aligned.toTranscriptome.out.bam", "rb").read()) == gzip.decompress(open(os.path.join(ref, "Aligned.toTranscriptome.out.bam"), "rb").read())
    if os.path.exists(os.path.join(ref, "_STARpass1/Log.final.out")):
        assert log_counters(out + "_STARpass1/Log.final.out") == log_counters(os.path.join(ref, "_STARpass1/Log.final.out"))
    if os.path.exists(os.path.join(ref, "_STARgenome/sha256.txt")):
        for line in open(os.path.join(ref, "_STARgenome/sha256.txt")):
            name, digest = line.split()
            assert hashlib.sha256(open(out + "_STARgenome/" + name, "rb").read()).hexdigest() == digest, name
