"""--outSAMtype BAM Unsorted (SURVEY.md §8f N1): the decompressed BAM stream of the host code (driven by the oracle engine on CPU)
must equal the unmodified reference's record for record; BGZF framing is checked structurally (block sizes, EOF marker).  No GPU."""
import ctypes as C
import gzip
import os
import struct
import subprocess

import pytest

import conftest as cf
import oracle_capi as oc

ROOT = cf.ROOT


def parse_bam(path):
    raw = open(path, "rb").read()
    return (raw,) + parse_bam_stream(gzip.decompress(raw))


def parse_bam_stream(d):
    """header text, references and records of a decompressed BAM stream"""
    assert d[:4] == b"BAM\x01"
    lt = struct.unpack("<i", d[4:8])[0]
    text = d[8:8 + lt]
    o = 8 + lt
    nref = struct.unpack("<i", d[o:o + 4])[0]
    o += 4
    refs = []
    for _ in range(nref):
        ln = struct.unpack("<i", d[o:o + 4])[0]
        refs.append((d[o + 4:o + 4 + ln], struct.unpack("<i", d[o + 4 + ln:o + 8 + ln])[0]))
        o += 8 + ln
    recs = []
    while o < len(d):
        bs = struct.unpack("<i", d[o:o + 4])[0]
        recs.append(d[o:o + 4 + bs])
        o += 4 + bs
    return text, refs, recs


def check_bgzf(raw):
    """every member is a BGZF block (gzip header with the BC extra field, total size <= 64 KB); the file ends with the EOF marker"""
    o, n = 0, 0
    while o < len(raw):
        assert raw[o:o + 4] == b"\x1f\x8b\x08\x04" and raw[o + 12:o + 14] == b"BC"
        bsize = struct.unpack("<H", raw[o + 16:o + 18])[0] + 1
        assert bsize <= 0x10000
        o += bsize
        n += 1
    assert o == len(raw)
    assert raw[-28:] == bytes([0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 0x42, 0x43, 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0])
    return n


def _header_lines(text):
    return [l for l in text.split(b"\n") if not l.startswith(b"@PG") and not l.startswith(b"@CO")]


def bam_summary(text, refs, recs):
    """header lines (without @PG / @CO), references, number and digest of the records: how refcmp.json stores a BAM file of the reference"""
    return {"header": [l.decode() for l in _header_lines(text)], "refs": [[n.decode(), ln] for n, ln in refs], "records": len(recs),
            "records_sha256": cf.sha256_lines(recs)}


CASES = [
    ("std", []),
    ("hard", []),
    ("se", []),
    ("std", ["--outSAMattributes", "NH", "HI", "AS", "nM", "NM", "MD", "jM", "jI", "MC", "XS", "--outSAMunmapped", "Within", "--outFilterMultimapNmax", "20"]),
    ("hard", ["--outSAMunmapped", "Within", "KeepPairs", "--outSAMattributes", "All", "--outSAMattrRGline", "ID:rg1", "SM:x", "--outSAMmode", "NoQS"]),
    ("hard", ["--alignEndsType", "EndToEnd", "--outSAMprimaryFlag", "AllBestScore", "--outSAMflagOR", "1024", "--outSAMattrIHstart", "0", "--outSAMmapqUnique", "60"]),
]


def input_files(golden, base):
    return [os.path.join(golden, base + "_1.fq")] + ([os.path.join(golden, base + "_2.fq")] if base != "se" else [])


@pytest.mark.parametrize("base,extra", CASES)
def test_bam_records_equal_the_reference(oracle, golden, refcmp, tmp_path, base, extra):
    """Against the reference's file (refcmp.json, written by the reference with --runThreadN 1)."""
    out = str(tmp_path) + "/"
    cmd = [oc.ORACLE_CLI, "--genomeDir", os.path.join(golden, "idx"), "--readFilesIn"] + input_files(golden, base) + ["--outFileNamePrefix", out,
           "--runThreadN", "3", "--outSAMtype", "BAM", "Unsorted"] + extra + ["--gpuChunkReads", "700"]
    subprocess.check_call(cmd, stdout=subprocess.DEVNULL, cwd=out)
    assert not os.path.exists(out + "Aligned.out.sam")
    raw, text, refs, recs = parse_bam(out + "Aligned.out.bam")
    assert check_bgzf(raw) >= 2
    assert bam_summary(text, refs, recs) == refcmp("bam", base, extra)["bam"]


def test_bam_record_count_and_names_match_the_sam_golden(oracle, golden, tmp_path):
    """Without the reference binary: the BAM of the std set has the same records (QNAME, FLAG, POS) as the committed SAM golden."""
    out = str(tmp_path) + "/"
    subprocess.check_call([oc.ORACLE_CLI, "--genomeDir", os.path.join(golden, "idx"), "--readFilesIn", os.path.join(golden, "std_1.fq"), os.path.join(golden, "std_2.fq"),
                           "--outFileNamePrefix", out, "--runThreadN", "2", "--outSAMtype", "BAM", "Unsorted", "--outBAMcompression", "6"], stdout=subprocess.DEVNULL)
    raw, text, refs, recs = parse_bam(out + "Aligned.out.bam")
    check_bgzf(raw)
    sam = cf.sam_body(os.path.join(golden, "ref_std", "Aligned.out.sam"))
    assert len(recs) == len(sam)
    for rec, line in zip(recs, sam):
        f = line.split(b"\t")
        refid, pos, bmn, fn = struct.unpack("<iiII", rec[4:20])
        lname = bmn & 0xff
        assert rec[36:36 + lname - 1] == f[0] and (fn >> 16) == int(f[1]) and pos + 1 == int(f[3]) and ((bmn >> 8) & 0xff) == int(f[4])


def test_sharded_bam_merge(oracle, lib, golden, tmp_path):
    world = 2
    pre = str(tmp_path) + "/m_"
    args = ["--genomeDir", os.path.join(golden, "idx"), "--readFilesIn", os.path.join(golden, "std_1.fq"), os.path.join(golden, "std_2.fq"), "--outSAMtype", "BAM", "Unsorted"]
    for r in range(world):
        subprocess.check_call([oc.ORACLE_CLI] + args + ["--outFileNamePrefix", pre + "shard%d." % r, "--gpuShardIndex", str(r), "--gpuShardCount", str(world)], stdout=subprocess.DEVNULL)
    argv = ["STAR"] + args + ["--outFileNamePrefix", pre]
    arr = (C.c_char_p * len(argv))(*[a.encode() for a in argv])
    lib.star_host_merge_shards.argtypes = [C.c_int, C.POINTER(C.c_char_p), C.c_int, C.c_void_p]
    assert lib.star_host_merge_shards(len(argv), arr, world, None) == 0
    whole = str(tmp_path) + "/w_"
    subprocess.check_call([oc.ORACLE_CLI] + args + ["--outFileNamePrefix", whole], stdout=subprocess.DEVNULL)
    a, b = parse_bam(pre + "Aligned.out.bam"), parse_bam(whole + "Aligned.out.bam")
    check_bgzf(a[0])
    assert a[2] == b[2] and a[3] == b[3]


def test_sharded_sorted_bam_merge(oracle, lib, golden, tmp_path):
    """Coordinate-sorted BAM of a sharded run: every shard leaves its records + sort keys, the merge sorts the whole run; equal to the
    single-process file record for record (Within: the unmapped records come last, in read order, across shards)."""
    world = 3
    pre = str(tmp_path) + "/m_"
    args = ["--genomeDir", os.path.join(golden, "idx"), "--readFilesIn", os.path.join(golden, "hard_1.fq"), os.path.join(golden, "hard_2.fq"),
            "--outSAMtype", "BAM", "Unsorted", "SortedByCoordinate", "--outSAMunmapped", "Within", "--runThreadN", "2"]
    for r in range(world):
        subprocess.check_call([oc.ORACLE_CLI] + args + ["--outFileNamePrefix", pre + "shard%d." % r, "--gpuShardIndex", str(r), "--gpuShardCount", str(world)], stdout=subprocess.DEVNULL)
    argv = ["STAR"] + args + ["--outFileNamePrefix", pre]
    arr = (C.c_char_p * len(argv))(*[a.encode() for a in argv])
    lib.star_host_merge_shards.argtypes = [C.c_int, C.POINTER(C.c_char_p), C.c_int, C.c_void_p]
    assert lib.star_host_merge_shards(len(argv), arr, world, None) == 0
    whole = str(tmp_path) + "/w_"
    subprocess.check_call([oc.ORACLE_CLI] + args + ["--outFileNamePrefix", whole], stdout=subprocess.DEVNULL)
    for f in ("Aligned.out.bam", "Aligned.sortedByCoord.out.bam"):
        a, b = parse_bam(pre + f), parse_bam(whole + f)
        check_bgzf(a[0])
        assert a[2] == b[2] and len(a[3]) == len(b[3]) and a[3] == b[3], f


SORT_CASES = [
    ("std", []),
    ("hard", ["--outSAMunmapped", "Within"]),
    ("se", ["--outSAMunmapped", "Within", "--outSAMattributes", "NH", "HI", "AS", "nM", "NM", "MD"]),
    ("hard", ["--outSAMunmapped", "Within", "KeepPairs", "--outFilterMultimapNmax", "20", "--winAnchorMultimapNmax", "100"]),
]


@pytest.mark.parametrize("base,extra", SORT_CASES)
def test_sorted_bam_equals_the_reference(oracle, golden, refcmp, tmp_path, base, extra):
    """--outSAMtype BAM Unsorted SortedByCoordinate: both files; the sorted one must list the same records in the same order as the
    reference's bin-sorted file (coordinate, then read order; unmapped reads last in read order), header with SO:coordinate.
    Reference files: refcmp.json, written by the reference with --runThreadN 2."""
    out = str(tmp_path) + "/"
    cmd = [oc.ORACLE_CLI, "--genomeDir", os.path.join(golden, "idx"), "--readFilesIn"] + input_files(golden, base) + ["--outFileNamePrefix", out,
           "--runThreadN", "3", "--outSAMtype", "BAM", "Unsorted", "SortedByCoordinate"] + extra + ["--gpuChunkReads", "500"]
    subprocess.check_call(cmd, stdout=subprocess.DEVNULL, cwd=out)
    ref = refcmp("sorted", base, extra)
    srt_o, uns_o = parse_bam(out + "Aligned.sortedByCoord.out.bam"), parse_bam(out + "Aligned.out.bam")
    check_bgzf(srt_o[0])
    assert srt_o[1].startswith(b"@HD\tVN:1.4\tSO:coordinate\n")
    assert bam_summary(*srt_o[1:]) == ref["sorted"]
    # the unsorted file next to it is unchanged by the extra output (the reference runs 2 threads here: compare as a multiset)
    assert bam_summary(uns_o[1], uns_o[2], sorted(uns_o[3])) == ref["unsorted_as_multiset"]
    keys = [struct.unpack("<II", r[4:12]) for r in srt_o[3]]
    assert keys == sorted(keys), "not coordinate-sorted"
