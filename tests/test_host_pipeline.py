"""CPU tests of the host side around the engine (the drop-in command line driven by the oracle engine): the three-stage chunk
pipeline, input errors in a late chunk, read sharding and the shard merge.  No GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import conftest as cf
import oracle_capi as oc

ROOT = cf.ROOT


def _cli(genome, files, out, extra=(), threads=3, check=True):
    cmd = [oc.ORACLE_CLI, "--genomeDir", genome, "--readFilesIn"] + files + ["--outFileNamePrefix", out, "--runThreadN", str(threads)] + list(extra)
    return subprocess.run(cmd, capture_output=True, text=True, timeout=300, check=check)


@pytest.mark.parametrize("chunk", [1, 7, 256, 5000])
def test_outputs_do_not_depend_on_the_chunk_size(oracle, golden, tmp_path, chunk):
    """Chunks flow through reader / engine / output threads with 3 buffers in flight: order and content must not change."""
    out = str(tmp_path) + "/"
    n = 300 if chunk < 256 else 0   # tiny chunks: a prefix of the reads is enough (and keeps the test short)
    extra = ["--gpuChunkReads", str(chunk)] + (["--readMapNumber", str(n)] if n else [])
    _cli(os.path.join(golden, "idx"), [os.path.join(golden, "std_1.fq"), os.path.join(golden, "std_2.fq")], out, extra)
    ref = cf.sam_body(os.path.join(golden, "ref_std", "Aligned.out.sam"))
    ours = cf.sam_body(out + "Aligned.out.sam")
    if n:   # the first n reads = the first n record names of the FASTQ
        with open(os.path.join(golden, "std_1.fq")) as f:
            lines = f.read().split("\n")
        keep = set(lines[4 * i][1:].split()[0].split("/")[0].encode() for i in range(n))
        ref = [l for l in ref if l.split(b"\t")[0] in keep]
    assert ours == ref


def test_input_error_in_a_late_chunk_stops_the_run(oracle, golden, tmp_path):
    """readLoad.cpp:66-71: quality length != sequence length is fatal; with the pipeline the error surfaces from the reader thread
    while earlier chunks are still being mapped / written — the process must exit with the reference's code, not hang."""
    with open(os.path.join(golden, "se_1.fq")) as f:
        lines = f.read().split("\n")
    bad = list(lines)
    rec = 150
    bad[4 * rec + 3] = bad[4 * rec + 3][:-3]           # truncate one quality string
    fq = str(tmp_path / "bad.fq")
    open(fq, "w").write("\n".join(bad))
    r = _cli(os.path.join(golden, "idx"), [fq], str(tmp_path) + "/o/", ["--gpuChunkReads", "64"], check=False)
    assert r.returncode != 0
    assert "quality string length is not equal to sequence length" in r.stderr
    assert "FATAL ERROR, exiting" in r.stderr


@pytest.mark.parametrize("piped", [False, True])
def test_text_that_is_not_a_record_is_fatal(oracle, golden, tmp_path, piped):
    """ReadAlignChunk_processChunks.cpp:192-207: at a record boundary only '@' / '>' start a record and only a blank / end of file ends the
    input; anything else is the reference's 'wrong read ID line format' error (exit 104), not a silent end of the input.  Both parsers
    (memory-mapped files; the stream parser behind --readFilesCommand)."""
    with open(os.path.join(golden, "se_1.fq")) as f:
        lines = f.read().split("\n")
    bad = lines[:4 * 100] + ["garbage that is not a record"] + lines[4 * 100:]
    fq = str(tmp_path / "bad.fq")
    open(fq, "w").write("\n".join(bad))
    extra = ["--gpuChunkReads", "64"] + (["--readFilesCommand", "cat"] if piped else [])
    r = _cli(os.path.join(golden, "idx"), [fq], str(tmp_path) + "/o/", extra, check=False)
    assert r.returncode == 104
    assert "wrong read ID line format" in r.stderr and "garbage that is not a record" in r.stderr


@pytest.mark.parametrize("world", [3])
def test_shards_partition_the_reads_in_order(oracle, golden, tmp_path, world):
    """--gpuShardIndex/--gpuShardCount: contiguous slices by record index, every read in exactly one shard, global read numbering kept."""
    bodies = []
    for r in range(world):
        out = str(tmp_path) + "/s%d." % r
        _cli(os.path.join(golden, "idx"), [os.path.join(golden, "se_1.fq")], out, ["--gpuShardIndex", str(r), "--gpuShardCount", str(world), "--outSAMreadID", "Number"])
        assert os.path.exists(out + "shard.bin") and not os.path.exists(out + "SJ.out.tab")
        sam = open(out + "Aligned.out.sam").read().split("\n")
        assert (sam[0].startswith("@")) == (r == 0)     # only shard 0 carries the header
        bodies.append(cf.sam_body(out + "Aligned.out.sam"))
    whole = str(tmp_path) + "/w."
    _cli(os.path.join(golden, "idx"), [os.path.join(golden, "se_1.fq")], whole, ["--outSAMreadID", "Number"])
    assert sum(bodies, []) == cf.sam_body(whole + "Aligned.out.sam")


def test_merge_without_allreduced_counters_sums_the_shard_files(oracle, lib, golden, tmp_path):
    """star_host_merge_shards(counters24 = NULL): the counters come from the shard files; outputs equal the single-process reference."""
    world = 2
    pre = str(tmp_path) + "/m_"
    args = ["--genomeDir", os.path.join(golden, "idx"), "--readFilesIn", os.path.join(golden, "std_1.fq"), os.path.join(golden, "std_2.fq")]
    for r in range(world):
        subprocess.check_call([oc.ORACLE_CLI] + args + ["--outFileNamePrefix", pre + "shard%d." % r, "--gpuShardIndex", str(r), "--gpuShardCount", str(world)],
                              stdout=subprocess.DEVNULL, timeout=300)
    argv = ["STAR"] + args + ["--outFileNamePrefix", pre]
    arr = (C.c_char_p * len(argv))(*[a.encode() for a in argv])
    lib.star_host_merge_shards.argtypes = [C.c_int, C.POINTER(C.c_char_p), C.c_int, C.c_void_p]
    assert lib.star_host_merge_shards(len(argv), arr, world, None) == 0
    ref = os.path.join(golden, "ref_std")
    assert cf.sam_body(pre + "Aligned.out.sam") == cf.sam_body(os.path.join(ref, "Aligned.out.sam"))
    assert open(pre + "SJ.out.tab", "rb").read() == open(os.path.join(ref, "SJ.out.tab"), "rb").read()
    assert cf.log_counters(pre + "Log.final.out") == cf.log_counters(os.path.join(ref, "Log.final.out"))


def _variant(lines, kind):
    out = list(lines)
    n = len(out) // 4
    if kind == "crlf":
        return "\r\n".join(out[:4 * n]) + "\r\n"
    if kind == "no_final_newline":
        return "\n".join(out[:4 * n])
    if kind == "trailing_blank_lines":
        return "\n".join(out[:4 * n]) + "\n\n\n"
    if kind == "comments_and_filter_flags":
        for r in range(n):
            out[4 * r] = out[4 * r].split()[0] + (" 1:Y:0:ACGT" if r % 3 == 0 else " 2:N:18:ACGT extra words")
            if r % 5 == 0:
                out[4 * r + 1] = out[4 * r + 1].lower()
        return "\n".join(out[:4 * n]) + "\n"
    raise ValueError(kind)


@pytest.mark.parametrize("kind", ["crlf", "no_final_newline", "trailing_blank_lines", "comments_and_filter_flags"])
def test_mapped_file_reader_equals_the_stream_reader(oracle, golden, tmp_path, kind):
    """Plain FASTQ files go through the memory-mapped parallel parser, piped input (--readFilesCommand) through the line-by-line stream
    parser (the restatement of processChunks/readLoad): same records, names, filter flags, order — on awkward but legal text."""
    files = []
    for m in (1, 2):
        with open(os.path.join(golden, "std_%d.fq" % m)) as f:
            lines = f.read().split("\n")
        while lines and lines[-1] == "":
            lines.pop()
        p = str(tmp_path / ("v_%d.fq" % m))
        with open(p, "w", newline="") as f:
            f.write(_variant(lines[:4 * 600], kind))
        files.append(p)
    extra = ["--gpuChunkReads", "97", "--outSAMunmapped", "Within", "--readNameSeparator", "/", "_"]
    a, b = str(tmp_path) + "/fast.", str(tmp_path) + "/stream."
    _cli(os.path.join(golden, "idx"), files, a, extra, threads=4)
    _cli(os.path.join(golden, "idx"), files, b, extra + ["--readFilesCommand", "cat"], threads=4)
    assert "reads input" in open(a + "Log.out").read()
    sa, sb_ = cf.sam_body(a + "Aligned.out.sam"), cf.sam_body(b + "Aligned.out.sam")
    assert len(sa) > 1000 and sa == sb_
    assert open(a + "SJ.out.tab", "rb").read() == open(b + "SJ.out.tab", "rb").read()
    assert cf.log_counters(a + "Log.final.out") == cf.log_counters(b + "Log.final.out")
    if kind == "comments_and_filter_flags":
        flags = [int(l.split(b"\t")[1]) for l in sa]
        assert any(f & 0x200 for f in flags) and not all(f & 0x200 for f in flags)


def _split_fastq(src, n_first, dst_a, dst_b):
    with open(src) as f:
        lines = f.read().split("\n")
    while lines and lines[-1] == "":
        lines.pop()
    open(dst_a, "w").write("\n".join(lines[:4 * n_first]) + "\n")
    open(dst_b, "w").write("\n".join(lines[4 * n_first:]) + "\n")


RG_MODES = ["plain", "command"]


def rg_header_lines(sam):
    return [l.decode() for l in open(sam, "rb").read().split(b"\n") if l.startswith(b"@RG")]


def rg_inputs(golden, tmp, mode):
    """mates split into two files each (700 + the rest) -> comma-separated lists, and the read-group options of the run"""
    parts = {}
    for m in (1, 2):
        a, b = os.path.join(str(tmp), "a_%d.fq" % m), os.path.join(str(tmp), "b_%d.fq" % m)
        _split_fastq(os.path.join(golden, "std_%d.fq" % m), 700, a, b)
        parts[m] = a + "," + b
    extra = ["--outSAMattrRGline", "ID:lane1", "SM:s1", ",", "ID:lane2", "SM:s1", "PL:x", "--outSAMunmapped", "Within", "--outSAMattributes", "NH", "HI", "AS", "nM", "RG"]
    if mode == "command":
        extra += ["--readFilesCommand", "cat"]
    return parts, extra


@pytest.mark.parametrize("mode", RG_MODES)
def test_comma_separated_file_lists_and_read_groups(oracle, golden, refcmp, tmp_path, mode):
    """--readFilesIn a1,a2 b1,b2 with one read group per file (--outSAMattrRGline ID:x , ID:y): records, RG tags, @RG header lines and
    counters equal the unmodified reference's (which concatenates the lists through a FIFO with FILE markers; refcmp.json)."""
    parts, extra = rg_inputs(golden, tmp_path, mode)
    out = str(tmp_path) + "/"
    subprocess.check_call([oc.ORACLE_CLI, "--genomeDir", os.path.join(golden, "idx"), "--readFilesIn", parts[1], parts[2], "--outFileNamePrefix", out,
                           "--runThreadN", "3"] + extra + ["--gpuChunkReads", "333"], stdout=subprocess.DEVNULL, cwd=out)
    ref = refcmp("rg", mode)
    assert cf.run_summary(out) == ref["outputs"]
    sam_o = cf.sam_body(out + "Aligned.out.sam")
    assert any(b"RG:Z:lane1" in l for l in sam_o) and any(b"RG:Z:lane2" in l for l in sam_o)
    assert rg_header_lines(out + "Aligned.out.sam") == ref["rg_header"] and len(ref["rg_header"]) == 2


def test_shards_over_a_file_list(oracle, golden, tmp_path):
    """sharding counts records across all files of a list: 3 shards over 2 files reproduce the unsharded output in order"""
    parts = []
    for m in (1, 2):
        a, b = str(tmp_path / ("a_%d.fq" % m)), str(tmp_path / ("b_%d.fq" % m))
        _split_fastq(os.path.join(golden, "std_%d.fq" % m), 450, a, b)
        parts.append(a + "," + b)
    bodies = []
    for r in range(3):
        out = str(tmp_path) + "/s%d." % r
        _cli(os.path.join(golden, "idx"), parts, out, ["--gpuShardIndex", str(r), "--gpuShardCount", "3", "--outSAMreadID", "Number"])
        bodies.append(cf.sam_body(out + "Aligned.out.sam"))
    whole = str(tmp_path) + "/w."
    _cli(os.path.join(golden, "idx"), parts, whole, ["--outSAMreadID", "Number"])
    assert all(len(b) > 0 for b in bodies) and sum(bodies, []) == cf.sam_body(whole + "Aligned.out.sam")


def test_parallel_line_index_of_a_large_file(oracle, golden, tmp_path):
    """The memory-mapped reader finds the lines of a chunk with several threads per mate (slices of >= 1 MB, ranges sized from the line
    length seen so far, a second range when the estimate was short).  A file of several MB with growing record lengths must give the
    same records as the stream parser (behind --readFilesCommand cat), across chunk boundaries."""
    with open(os.path.join(golden, "std_1.fq")) as f:
        l1 = f.read().split("\n")
    with open(os.path.join(golden, "std_2.fq")) as f:
        l2 = f.read().split("\n")
    nrec = min(len(l1), len(l2)) // 4
    big1, big2 = [], []
    k = 0
    while sum(len(x) for x in big1) < 5_000_000:       # the records repeated under new names; later copies get longer ID lines
        for r in range(nrec):
            pad = " pad" * (k // 2000)
            big1 += ["@n%d%s" % (k, pad), l1[4 * r + 1], "+", l1[4 * r + 3]]
            big2 += ["@n%d%s" % (k, pad), l2[4 * r + 1], "+", l2[4 * r + 3]]
            k += 1
    f1, f2 = str(tmp_path / "big_1.fq"), str(tmp_path / "big_2.fq")
    open(f1, "w").write("\n".join(big1))               # (no newline at the end of mate 1)
    open(f2, "w").write("\n".join(big2) + "\n")
    outs = []
    for tag, extra, thr in (("map", [], 8), ("stream", ["--readFilesCommand", "cat"], 2)):
        out = str(tmp_path) + "/" + tag + "/"
        os.makedirs(out)
        _cli(os.path.join(golden, "idx"), [f1, f2], out, ["--gpuChunkReads", "9000", "--readMapNumber", "30000"] + extra, threads=thr)
        outs.append(cf.sam_body(out + "Aligned.out.sam"))
    assert len(outs[0]) > 30000 and outs[0] == outs[1]


@pytest.mark.parametrize("pct", [125, 40])
def test_page_locked_chunk_buffers_and_second_fetch(oracle, golden, tmp_path, pct):
    """With an engine that offers page-locked memory (star_gpu_host_alloc) the driver sizes the record buffer for 5/4 records per read,
    copies the sequences through a page-locked block, and fetches the results a second time (star_gpu_download_results) into a larger
    buffer when a chunk holds more records.  The optional vtable members are emulated around the oracle engine (STAR_CLI_PINNED_EMUL);
    a buffer of 0.4 records per read forces the second fetch in every chunk.  Output = the reference's."""
    out = str(tmp_path) + "/"
    env = dict(os.environ, STAR_CLI_PINNED_EMUL="1", STAR_B200_PINNED_ALIGNS_PCT=str(pct))
    cmd = [oc.ORACLE_CLI, "--genomeDir", os.path.join(golden, "idx"), "--readFilesIn", os.path.join(golden, "std_1.fq"), os.path.join(golden, "std_2.fq"),
           "--outFileNamePrefix", out, "--runThreadN", "3", "--gpuChunkReads", "333"]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-1000:]
    note = [l for l in r.stderr.split("\n") if l.startswith("pinned emulation:")][0].split()
    allocs, misses = int(note[2]), int(note[5])
    assert allocs >= 3 and (misses > 0) == (pct < 100), note
    ref = os.path.join(golden, "ref_std")
    assert cf.sam_body(out + "Aligned.out.sam") == cf.sam_body(os.path.join(ref, "Aligned.out.sam"))
    assert open(out + "SJ.out.tab", "rb").read() == open(os.path.join(ref, "SJ.out.tab"), "rb").read()
    assert cf.log_counters(out + "Log.final.out") == cf.log_counters(os.path.join(ref, "Log.final.out"))


def test_host_stage_threads_follow_the_cpu_allowance(oracle, golden, tmp_path):
    """The reader and the formatter run next to the thread that drives the GPU: each uses min(--runThreadN, 32, CPUs allowed / 2) threads
    (affinity mask and cgroup quota, not the logical CPUs the process sees), or STAR_B200_HOST_STAGE_THREADS; Log.out reports the number
    and the output does not depend on it."""
    import re
    outs = []
    for tag, env_extra, thr in (("a", {}, 64), ("b", {"STAR_B200_HOST_STAGE_THREADS": "3"}, 64), ("c", {}, 1)):
        out = str(tmp_path) + "/" + tag + "/"
        os.makedirs(out)
        cmd = [oc.ORACLE_CLI, "--genomeDir", os.path.join(golden, "idx"), "--readFilesIn", os.path.join(golden, "std_1.fq"), os.path.join(golden, "std_2.fq"),
               "--outFileNamePrefix", out, "--runThreadN", str(thr), "--gpuChunkReads", "700"]
        subprocess.run(cmd, env=dict(os.environ, **env_extra), capture_output=True, text=True, timeout=300, check=True)
        m = re.search(r"host stages used (\d+) threads each \(--runThreadN (\d+), CPUs allowed to this process (\d+)\)", open(out + "Log.out").read())
        assert m, "no thread report in Log.out"
        used, asked, allowed = int(m.group(1)), int(m.group(2)), int(m.group(3))
        assert asked == thr and 1 <= allowed <= (os.cpu_count() or 1)
        if tag == "a":
            assert used == max(2, min(32, allowed // 2, thr)) or used == min(thr, max(2, min(32, allowed // 2)))
        elif tag == "b":
            assert used == 3
        else:
            assert used == 1
        outs.append(cf.sam_body(out + "Aligned.out.sam"))
    assert outs[0] == outs[1] == outs[2]
