#!/usr/bin/env python3
"""bench.py — throughput of the STAR alignment hot path on B200 (contract: see the task statement / DESIGN.md §5).

A "step" = one pass of the whole hot path (prep -> MMP seed search -> windows -> stitch/extend -> select -> pack) over
one chunk of synthetic 2x100 bp read pairs.

  value   : read pairs / s with the chunk already resident in HBM (star_gpu_upload_chunk once, star_gpu_map_resident per step)
  e2e     : the same metric through the reference-facing C-ABI call star_gpu_map_chunk with PINNED HOST buffers
            (host->device copy of the sequences and device->host copy of all results inside the timed region)
  cli_e2e : the drop-in command line star_b200/bin/STAR, FASTQ files -> Aligned.out.sam, wall clock minus a
            --readMapNumber 1 (start-up + index load) run — the same scope and the same files as the reference arm
  roofline: MMP seed-search stage, algorithmic bytes (SURVEY.md §8d formula, counts from the instrumented ORACLE on a
            sample) / CUDA-event duration of that stage
  parity_sample: the engine's records for the first pairs of the timed chunk compared field by field with the oracle's
            (the run FAILS on a difference)
  cpu_baseline: the UNMODIFIED reference (oracle/_ref/STAR) on all host cores on a bounded sample of the same workload

Workload (BASELINE.json configs[1]): no real genome exists here or on the GPU box and there is no network (SURVEY.md F7),
so the genome is the survey's self-contained tier scaled to GRCh38: 24 chromosomes with the GRCh38 lengths (3.09 Gb),
repeat families, N blocks, ~27 k genes / ~350 k annotated junctions (tools/synth.py preset "grch38"), index
(Genome 3.2 GB, SA 24 GB, SAindex 1.6 GB; --genomeSAindexNbases 14, --sjdbOverhang 99) built ONCE per box by this
repository's own `--runMode genomeGenerate` on the GPU and cached under the work directory; both arms load that
directory.  `--preset chr21` selects the 46.7 Mb genome of round 1 (index built by the reference's genomeGenerate when
oracle/_ref/STAR was built, otherwise by this repository's, which writes the same files).

--dump-outputs DIR writes the read results and alignment records of the last timed step of the value leg for a fixed, seeded
sample of the reads (dump_outputs): the inputs depend only on the arguments, so two builds can be compared output for output.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--preset grch38|chr21] [--mm 0.005] [--read-len 100]
                  [--dump-outputs DIR]
  torchrun --nproc-per-node N bench.py --gpus N ...      (one rank per GPU; reads are sharded, weak scaling)
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True   # the tree may be read-only: the modules imported from tools/ and tests/ leave no bytecode there
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
REF_STAR = os.path.join(ROOT, "oracle", "_ref", "STAR")
OUR_STAR = os.path.join(ROOT, "star_b200", "bin", "STAR")
METRIC = "reads/sec (2x100 bp PE)"
UNIT = "read pairs/s"
SAINDEX_NBASES = {"tiny": 7, "small": 9, "chr21": 11, "grch38_8th": 13, "grch38": 14}
DUMP_READS = 32768       # --dump-outputs: size of the fixed sample of reads
DUMP_BYTES = 63 << 20    # and the most data it writes (with the .npy headers: < 64 MB)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def workload_name(preset, read_len, mm):
    g = {"grch38": "synthetic GRCh38-sized genome (3.09 Gb, 24 chr with the GRCh38 lengths, repeat families, ~350 k annotated junctions, sjdbOverhang 99, SAindexNbases 14; index ~29 GB)",
         "grch38_8th": "synthetic 1/8-scale GRCh38 model (386 Mb, 24 chr, sjdbOverhang 99, SAindexNbases 13)",
         "chr21": "synthetic chr21-sized genome (46.7 Mb, 3 chr, sjdbOverhang 99, SAindexNbases 11)"}.get(preset, "synthetic %s genome" % preset)
    return "%s, 2x%d bp PE, %.1f%% subst" % (g, read_len, mm * 100)


def allowed_cpus():
    """CPUs this process may use: the affinity mask, limited by the cgroup CPU quota (v2 cpu.max, v1 cfs_quota / cfs_period)."""
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        pass
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = min(n, max(1, -(-int(q) // int(p))))
    except (OSError, ValueError):
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0 and p > 0:
                n = min(n, max(1, -(-q // p)))
        except (OSError, ValueError):
            pass
    return n


def prepare_genome(workdir, preset, device=0, own_generate=False):
    """genome.fa + annot.gtf + idx/ under workdir (built once, cached).  Returns (chrs, trs, idx_dir, build_info).

    The index is built by the reference's generator for the small presets when oracle/_ref/STAR was built, otherwise by this repository's
    GPU generator, which writes the same files (tests/test_gpu_config_gate.py checks them against the reference's digests)."""
    import synth
    t0 = time.time()
    chrs = synth.make_genome(preset)
    trs = synth.make_annotation(chrs, preset)
    log("synthetic genome %s: %.1f s" % (preset, time.time() - t0))
    idx = os.path.join(workdir, "idx")
    info_path = os.path.join(idx, "build_info.json")
    if not os.path.exists(info_path):
        shutil.rmtree(idx, ignore_errors=True)
        os.makedirs(idx)
        t0 = time.time()
        synth.write_fasta(chrs, os.path.join(workdir, "genome.fa"))
        synth.write_gtf(chrs, trs, os.path.join(workdir, "annot.gtf"))
        t_files = time.time() - t0
        big = (own_generate or bool(synth.PRESETS[preset].get("big")) or os.environ.get("STAR_B200_BENCH_OWN_GENERATE") == "1"
               or not os.path.exists(REF_STAR))
        threads = str(min(64, os.cpu_count() or 8))
        args = ["--runMode", "genomeGenerate", "--genomeDir", "idx", "--genomeFastaFiles", "genome.fa", "--sjdbGTFfile", "annot.gtf",
                "--sjdbOverhang", "99", "--genomeSAindexNbases", str(SAINDEX_NBASES[preset]), "--runThreadN", threads, "--outFileNamePrefix", "gen_"]
        t0 = time.time()
        if big:   # the reference's generator needs ~1 h and ~32 GB for this size: the index is built by this repository's GPU generator
            subprocess.check_call([OUR_STAR] + args + ["--gpuDevice", str(device)], cwd=workdir, stdout=subprocess.DEVNULL)
            builder = "star_b200 --runMode genomeGenerate (GPU suffix sort)"
        else:
            subprocess.check_call([REF_STAR] + args, cwd=workdir, stdout=subprocess.DEVNULL)
            builder = "reference --runMode genomeGenerate"
        info = {"builder": builder, "seconds": round(time.time() - t0, 1), "fasta_gtf_seconds": round(t_files, 1)}
        try:
            info["phases"] = [l.strip() for l in open(os.path.join(workdir, "gen_Log.out")) if l.strip().startswith("[")]
        except OSError:
            pass
        json.dump(info, open(info_path, "w"))
        log("index built in %.1f s by %s" % (info["seconds"], builder))
    return chrs, trs, idx, json.load(open(info_path))


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
                  "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        self.gpu = gpu_index
        self.samples = []
        self.stop_flag = False
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.samples.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        for s in self.samples:
            try:
                sm.append(float(s[1]))
                mx = max(mx, float(s[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


class ReferenceRunner:
    """The unmodified reference on FASTQ files -> Aligned.out.sam, timed without its index load.

    Preferred: the index is put into SysV shared memory once (`--genomeLoad LoadAndExit`, the reference's own feature) and every run
    attaches to it (`LoadAndKeep`), so a run's wall clock is start-up + mapping + output; a `--readMapNumber 1` run is subtracted
    (SURVEY.md §8d).  Fallback when shared memory is refused: wall clock of a private-load run minus a private-load `--readMapNumber 1`
    run (measured once)."""

    def __init__(self, workdir, idx, threads):
        self.workdir, self.idx, self.threads = workdir, idx, threads
        self.shm = False
        self.t_load = None
        self.base = None

    def _run(self, fq1, fq2, tag, extra):
        out = os.path.join(self.workdir, tag)
        shutil.rmtree(out, ignore_errors=True)
        os.makedirs(out)
        t0 = time.time()
        subprocess.check_call([REF_STAR, "--genomeDir", self.idx, "--readFilesIn", fq1, fq2, "--outFileNamePrefix", out + "/", "--runThreadN", str(self.threads),
                               "--outSAMtype", "SAM"] + extra, stdout=subprocess.DEVNULL)
        dt = time.time() - t0
        return dt, out

    def start(self, fq1, fq2):
        if os.environ.get("STAR_B200_BENCH_NO_SHM") != "1":
            t0 = time.time()
            rc = subprocess.call([REF_STAR, "--genomeDir", self.idx, "--genomeLoad", "LoadAndExit", "--outFileNamePrefix", os.path.join(self.workdir, "shmload_")],
                                 stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            self.t_load = time.time() - t0
            self.shm = rc == 0
            if not self.shm:
                subprocess.call([REF_STAR, "--genomeDir", self.idx, "--genomeLoad", "Remove", "--outFileNamePrefix", os.path.join(self.workdir, "shmrm_")],
                                stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        self.extra = ["--genomeLoad", "LoadAndKeep"] if self.shm else []
        dt0, out0 = self._run(fq1, fq2, "ref_base", self.extra + ["--readMapNumber", "1"])
        shutil.rmtree(out0, ignore_errors=True)
        self.base = dt0
        log("reference: index %s, start-up/load-only run %.2f s" % ("in shared memory (loaded in %.1f s)" % self.t_load if self.shm else "loaded privately by every run", dt0))

    def run(self, fq1, fq2, keep=False):
        dt, out = self._run(fq1, fq2, "ref_run", self.extra)
        if not keep:
            shutil.rmtree(out, ignore_errors=True)
        return max(1e-3, dt - self.base), dt, out

    def stop(self):
        if self.shm:
            subprocess.call([REF_STAR, "--genomeDir", self.idx, "--genomeLoad", "Remove", "--outFileNamePrefix", os.path.join(self.workdir, "shmrm_")],
                            stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)

    def describe(self):
        return ("index in SysV shared memory (--genomeLoad LoadAndKeep), wall clock minus a --readMapNumber 1 run" if self.shm
                else "wall clock of the full run minus a --readMapNumber 1 (index load) run")


def cli_run(idx, fq1, fq2, out, threads, extra, device):
    shutil.rmtree(out, ignore_errors=True)
    os.makedirs(out)
    t0 = time.time()
    subprocess.check_call([OUR_STAR, "--genomeDir", idx, "--readFilesIn", fq1, fq2, "--outFileNamePrefix", out + "/", "--runThreadN", str(threads),
                           "--outSAMtype", "SAM", "--gpuDevice", str(device)] + extra, stdout=subprocess.DEVNULL)
    return time.time() - t0


def dump_outputs(path, res, al):
    """--dump-outputs: what a caller of the timed path receives (the read results and their alignment records) for a fixed, seeded
    sample of the reads, every field as <path>/result_<field>.npy and <path>/align_<field>.npy (float32 where that is exact, float64
    otherwise; records in read order), and the sampled read indices as <path>/sample_reads.npy.  The sample is cut short where the
    records would take it past DUMP_BYTES."""
    import star_b200 as sb
    as_float = lambda x: x.astype(np.float32 if x.dtype.itemsize <= 2 else np.float64)
    sample = np.sort(np.random.default_rng(20260917).choice(len(res), size=min(len(res), DUMP_READS), replace=False))
    rec_bytes = sum(as_float(np.zeros(1, sb.capi.ALIGN_DTYPE)[f]).nbytes for f in sb.capi.ALIGN_DTYPE.names)
    res_bytes = 8 * (len(sb.capi.RESULT_DTYPE.names) + 1)   # float64 fields + the index in sample_reads
    n_tr = res["nTrOut"][sample].astype(np.int64)
    sample = sample[np.cumsum(res_bytes + n_tr * rec_bytes) <= DUMP_BYTES]
    r = res[sample]
    recs = al[np.concatenate([np.arange(o, o + k, dtype=np.int64) for o, k in zip(r["trOffset"], r["nTrOut"])] + [np.zeros(0, np.int64)])]
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "sample_reads.npy"), sample.astype(np.float64))
    for f in sb.capi.RESULT_DTYPE.names:
        np.save(os.path.join(path, "result_%s.npy" % f), as_float(r[f]))
    for f in sb.capi.ALIGN_DTYPE.names:
        np.save(os.path.join(path, "align_%s.npy" % f), as_float(recs[f]))
    log("outputs of the last timed step: %d sampled reads, %d records -> %s" % (len(sample), len(recs), path))


def sam_records(path):
    with open(path, "rb") as f:
        return [l for l in f.read().split(b"\n") if l and not l.startswith(b"@")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pairs", type=int, default=int(os.environ.get("STAR_B200_BENCH_PAIRS", 1 << 20)), help="read pairs per GPU per step")
    ap.add_argument("--ref-pairs", type=int, default=int(os.environ.get("STAR_B200_BENCH_REF_PAIRS", 1 << 20)),
                    help="pairs of the chunk written as FASTQ for the reference / command-line legs")
    ap.add_argument("--ref-repeat", type=int, default=int(os.environ.get("STAR_B200_BENCH_REF_REPEAT", 2)),
                    help="the reference maps this many concatenated copies of the sample per step (round 1, 128-core box: 124-129 k pairs/s for 2 M, 4 M and 16 M pairs alike - it is bound by its serial FASTQ chunker, so the bounded sample is representative)")
    ap.add_argument("--cli-repeat", type=int, default=int(os.environ.get("STAR_B200_BENCH_CLI_REPEAT", 24)), help="copies of the sample mapped by the command-line leg")
    ap.add_argument("--preset", default=os.environ.get("STAR_B200_BENCH_PRESET", "grch38"))
    ap.add_argument("--mm", type=float, default=0.005)
    ap.add_argument("--read-len", type=int, default=100)
    ap.add_argument("--parity-pairs", type=int, default=20000)
    ap.add_argument("--no-cli", action="store_true", help="skip the command-line leg")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--workdir", default=os.environ.get("STAR_B200_BENCH_DIR", "/tmp/star_b200_bench"))
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step (value leg) for a fixed sample of the reads as DIR/<name>.npy (rank 0)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    import synth
    # If the GRCh38-sized index cannot be built on this box (it never falls back silently: config.workload names what ran and
    # config.fallback says why), both arms use the chr21-sized genome.  The first arm that fails leaves a marker for the other one.
    fail_marker = os.path.join(a.workdir, a.preset, "BUILD_FAILED")
    fallback = None
    if a.preset == "grch38" and os.environ.get("STAR_B200_BENCH_NO_FALLBACK") != "1":
        if os.path.exists(fail_marker):
            fallback = open(fail_marker).read().strip()
        elif rank == 0 and not os.path.exists(os.path.join(a.workdir, a.preset, "idx", "build_info.json")):
            try:
                os.makedirs(os.path.join(a.workdir, a.preset), exist_ok=True)
                prepare_genome(os.path.join(a.workdir, a.preset), a.preset, local_rank)
            except Exception as e:   # noqa: BLE001
                fallback = "GRCh38-sized index build failed on this box: %s" % str(e)[:300]
                shutil.rmtree(os.path.join(a.workdir, a.preset, "idx"), ignore_errors=True)
                open(fail_marker, "w").write(fallback)
                log("FALLBACK: " + fallback)
        if world > 1:   # the other ranks learn the outcome from the marker after rank 0 is done (file system, before any collective)
            t_wait = time.time()
            while rank != 0 and not (os.path.exists(fail_marker) or os.path.exists(os.path.join(a.workdir, a.preset, "idx", "build_info.json"))) and time.time() - t_wait < 1700:
                time.sleep(2)
            if os.path.exists(fail_marker):
                fallback = open(fail_marker).read().strip()
        if fallback:
            a.preset = "chr21"
    workdir = os.path.join(a.workdir, a.preset)
    os.makedirs(workdir, exist_ok=True)
    workload = workload_name(a.preset, a.read_len, a.mm)
    host_cores = os.cpu_count() or 1
    cpus_allowed = allowed_cpus()   # cgroup quota: the GPU boxes of round 2 show 128 logical CPUs and allow 16 (cpu.max = 1600000 100000)
    n = a.pairs
    config = {"workload": workload, "fallback": fallback, "pairs_per_gpu_per_step": n, "read_definition": "one 2x%d pair = one read (STAR 'Number of input reads')" % a.read_len,
              "reads": "tools/synth.py make_reads seed 1000 + rank: 50 % from annotated transcripts, 50 % from the genome, fragment 300"}
    tag = "" if (a.read_len == 100 and a.mm == 0.005) else "_L%d_mm%g" % (a.read_len, a.mm)

    # ------------------------------------------------------------------ reference arm
    if a.impl == "reference":
        if rank != 0:
            return 0
        chrs, trs, idx, build = prepare_genome(workdir, a.preset, 0)
        rp = min(a.ref_pairs, n)
        m1, m2 = synth.make_reads(chrs, trs, n, read_len=a.read_len, mm=a.mm, seed=1000)   # the chunk of our arm's rank 0
        fq1, fq2 = os.path.join(workdir, "cpu%s_1.fq" % tag), os.path.join(workdir, "cpu%s_2.fq" % tag)
        synth.write_fastq(m1[:rp], fq1)
        synth.write_fastq(m2[:rp], fq2)
        del m1, m2, chrs
        rep = max(1, a.ref_repeat)
        f1, f2 = ",".join([fq1] * rep), ",".join([fq2] * rep)
        rr = ReferenceRunner(workdir, idx, host_cores)
        rr.start(f1, f2)
        times = []
        try:
            for s in range(a.warmup + a.steps):
                dt, wall, _ = rr.run(f1, f2)
                if s >= a.warmup:
                    times.append(dt)
                log("reference step %d: %.2f s wall, %.2f s without start-up" % (s, wall, dt))
        finally:
            rr.stop()
        t = float(np.mean(times))
        v = rp * rep / t
        sample = "%d x the first %d pairs of the step's chunk per step, oracle/_ref/STAR --runThreadN %d --outSAMtype SAM, %s" % (rep, rp, host_cores, rr.describe())
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/int64", "data": "synthetic",
                "config": dict(config, reference_sample_pairs_per_step=rp * rep, threads=host_cores, index_build=build),
                "cpu_baseline": {"value": v, "unit": UNIT, "cores": host_cores, "cpus_allowed_by_cgroup": cpus_allowed, "kind": "reference", "sample": sample},
                "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
        return 0

    # ------------------------------------------------------------------ our arm
    import torch
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    if rank == 0:
        chrs, trs, idx, build = prepare_genome(workdir, a.preset, local_rank)
    if world > 1:
        dist.barrier()
    if rank != 0:
        chrs, trs, idx, build = prepare_genome(workdir, a.preset, local_rank)

    import star_b200 as sb
    lib = sb.load_library()
    t0 = time.time()
    index = sb.Index(lib, idx)
    t_index_host = time.time() - t0
    m1, m2 = synth.make_reads(chrs, trs, n, read_len=a.read_len, mm=a.mm, seed=1000 + rank)
    del chrs
    seq, off, _, nm = sb.pack_reads([m1, m2])
    t0 = time.time()
    eng = sb.Engine(lib, index, max_reads=n, device=local_rank)
    t_engine_init = time.time() - t0
    # pinned host buffers for the e2e leg
    pin_seq = torch.empty(seq.nbytes, dtype=torch.uint8, pin_memory=True)
    pin_seq.numpy()[:] = seq
    pin_off = torch.empty(off.nbytes, dtype=torch.uint8, pin_memory=True)
    pin_off.numpy().view(np.uint64)[:] = off
    pin_res = torch.empty(n * sb.capi.RESULT_DTYPE.itemsize, dtype=torch.uint8, pin_memory=True)
    pin_al = torch.empty(n * 2 * sb.capi.ALIGN_DTYPE.itemsize, dtype=torch.uint8, pin_memory=True)   # 2 alignments / read of head-room
    res_np = pin_res.numpy().view(sb.capi.RESULT_DTYPE)
    al_np = pin_al.numpy().view(sb.capi.ALIGN_DTYPE)
    ab = sb.capi.AlignBatch()
    ab.reads = res_np.ctypes.data
    ab.aligns = al_np.ctypes.data
    ab.alignsCapacity = al_np.shape[0]
    seq_p = pin_seq.numpy()
    off_p = pin_off.numpy().view(np.uint64)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- value: chunk resident in HBM
    eng.upload(seq_p, off_p, n, nm)
    for _ in range(a.warmup):
        eng.map_resident()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = lib.star_gpu_launch_count()
    sync_all()
    t0 = time.perf_counter()
    dev_ms, seed_ms, stitch_ms = 0.0, 0.0, 0.0
    last = None
    for _ in range(a.steps):
        st = eng.map_resident()
        dev_ms += st.ms_total
        seed_ms += st.ms_seed
        stitch_ms += st.ms_stitch
        last = st
    sync_all()
    wall = time.perf_counter() - t0
    launches = lib.star_gpu_launch_count() - launches0
    if a.dump_outputs and rank == 0:   # outside the timed region; the e2e leg below overwrites these buffers
        dump_outputs(a.dump_outputs, *eng.download(n, out=(res_np, al_np, ab)))
    # ---- e2e: host buffers through star_gpu_map_chunk
    for _ in range(max(1, a.warmup // 2)):
        eng.map_chunk(seq_p, off_p, n, nm, out=(res_np, al_np, ab))
    sync_all()
    t0 = time.perf_counter()
    h2d = d2h = 0
    n_al = 0
    for _ in range(a.steps):
        _, al_out, st2 = eng.map_chunk(seq_p, off_p, n, nm, out=(res_np, al_np, ab))
        h2d, d2h = st2.h2d_bytes, st2.d2h_bytes
        n_al = len(al_out)
    sync_all()
    wall_e2e = time.perf_counter() - t0
    clocks = sampler.finish()

    # max over ranks (device timing) and the single collective of the path: the Log.final.out counters (SURVEY.md §8e)
    t_val = max(dev_ms / 1e3, 0.0)
    if world > 1:
        tt = torch.tensor([t_val, wall, wall_e2e], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_val, wall, wall_e2e = [float(x) for x in tt.tolist()]
        counters = torch.tensor([n * a.steps, int((res_np["unmapType"] < 0).sum())], dtype=torch.int64, device="cuda")
        dist.all_reduce(counters)
    total_pairs = n * world * a.steps
    value = total_pairs / t_val
    e2e_value = total_pairs / wall_e2e
    rc_exit = 0

    if rank == 0:
        # ---- parity sample + algorithmic byte counts: the ORACLE on the first pairs of this step's chunk (checker only)
        peak_gbs, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(pk):
            peak_gbs, peak_src = float(json.load(open(pk))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        gstrand = int(index.view.contents.GstrandBit)
        w_sai, w_sa = (gstrand + 3) / 8.0, (gstrand + 1) / 8.0
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_capi as oc
        ns = min(n, a.parity_pairs)
        oe = oc.OracleEngine(oc.load_oracle(), index)
        t0 = time.perf_counter()
        res_o, al_o, st_o = oe.map_chunk(seq[: int(off[ns * 2])].copy(), off[: ns * 2 + 1].copy(), ns, nm)
        t_oracle = time.perf_counter() - t0
        oe.close()
        n_al_s = int(res_np["nTrOut"][:ns].sum())   # records are packed in read order: the first ns reads own the first n_al_s records
        res_g = res_np[:ns].copy()
        al_g = al_np[:n_al_s].copy()
        diffs = oc.compare_outputs(res_o, al_o, res_g, al_g)
        parity = {"pairs": ns, "alignments": int(len(al_o)), "diffs": len(diffs), "checker": "oracle/star_oracle.cpp (pinned to the reference), every field of every record"}
        if diffs:
            parity["first"] = diffs[:3]
            log("PARITY FAILURE on the bench chunk:\n" + "\n".join(diffs[:10]))
            rc_exit = 3
        b_pair_oracle = (st_o.mmp_sai_words * w_sai + st_o.mmp_compare_calls * w_sa + st_o.mmp_bases_examined * 1.0) / ns
        seed_s = seed_ms / a.steps / 1e3
        achieved = b_pair_oracle * n / seed_s / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "seed_kernel_traffic.json")
        if os.path.exists(tpath):
            try:
                tj = json.load(open(tpath))
                if int(tj.get("pairs_per_launch", -1)) == n and tj.get("preset") == a.preset and tj.get("read_len", 100) == a.read_len:
                    import hashlib
                    hh = hashlib.sha1()
                    for fsrc in ("seed_keyed.cuh", "seed_warp.cuh", "seed_types.cuh"):   # the capture is only valid for the kernel sources it was taken from
                        hh.update(open(os.path.join(ROOT, "star_b200", "csrc", "engine", fsrc), "rb").read())
                    l2 = int(os.environ.get("STAR_B200_L2_FETCH_BYTES", "64"))
                    if tj.get("kernel_sources_sha1") == hh.hexdigest() and int(tj.get("l2_fetch_bytes", 64)) == l2:
                        traffic = tj.get("dram_bytes_per_launch")
            except Exception:
                pass
        roofline = {"bound": "hbm", "kernel": "MMP seed search (all kernels between the prep and the window stage)", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
                    "frac": achieved / peak_gbs, "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_pair": b_pair_oracle,
                    "algorithmic_counts_per_pair": {"searches": st_o.mmp_searches / ns, "sai_words": st_o.mmp_sai_words / ns, "compare_calls": st_o.mmp_compare_calls / ns,
                                                    "bases": st_o.mmp_bases_examined / ns},
                    "kernel_ms": seed_s * 1e3, "stitch_kernel_ms": stitch_ms / a.steps}
        # ---- reference on the host cores + our command line, on the same FASTQ files
        cpu = None
        cli = None
        if world == 1 and not (a.no_cpu and a.no_cli):
            rp = min(a.ref_pairs, n)
            fq1, fq2 = os.path.join(workdir, "cpu%s_1.fq" % tag), os.path.join(workdir, "cpu%s_2.fq" % tag)
            synth.write_fastq(m1[:rp], fq1)
            synth.write_fastq(m2[:rp], fq2)
            if not a.no_cpu and os.path.exists(REF_STAR):
                rep = max(1, a.ref_repeat)
                f1, f2 = ",".join([fq1] * rep), ",".join([fq2] * rep)
                rr = ReferenceRunner(workdir, idx, host_cores)
                rr.start(f1, f2)
                try:
                    dt, wall_ref, _ = rr.run(f1, f2)
                finally:
                    rr.stop()
                cpu = {"value": rp * rep / dt, "unit": UNIT, "cores": host_cores, "cpus_allowed_by_cgroup": cpus_allowed, "kind": "reference",
                       "sample": "%d x the first %d pairs of the step's chunk, oracle/_ref/STAR --runThreadN %d --outSAMtype SAM, %s (%.2f s - %.2f s)"
                                 % (rep, rp, host_cores, rr.describe(), wall_ref, rr.base),
                       "oracle_port_1thread_pairs_per_s": ns / t_oracle}
            elif not a.no_cpu:
                cpu = {"value": ns / t_oracle, "unit": UNIT, "cores": 1, "kind": "port", "sample": "%d pairs, oracle/star_oracle.cpp, 1 thread" % ns}
            if not a.no_cli:
                eng.close()   # the command line creates its own context on this GPU
                eng = None
                rep = max(1, a.cli_repeat)
                f1, f2 = ",".join([fq1] * rep), ",".join([fq2] * rep)
                # --runThreadN of OUR command line: its reader, formatter and writer stages each use up to that many threads next to the engine thread.
                # Measured on the 128-core box (profiles/r02g_cli_threads.txt): every stage is faster with 32 than with 64 (engine 121 / 159 ms per
                # chunk, formatting 145 / 172, reader 115 / 155, writes 77 / 125) and much slower with 112: the stages compete for the cores.
                threads = max(8, min(32, host_cores // 4))
                t_base = cli_run(idx, f1, f2, os.path.join(workdir, "cli_base"), threads, ["--readMapNumber", "1"], local_rank)
                t_full = cli_run(idx, f1, f2, os.path.join(workdir, "cli_run"), threads, [], local_rank)
                host_lines = []
                try:
                    host_lines = [l.strip() for l in open(os.path.join(workdir, "cli_run", "Log.out")) if l.startswith("star-b200:")]
                except OSError:
                    pass
                pass_wall = None   # the command line's own clock around its mapping pass (cross-check of wall minus start-up: the index load alone varies by seconds)
                for l in host_lines:
                    if "mapping pass wall" in l:
                        try:
                            pass_wall = float(l.split("mapping pass wall")[1].split("ms")[0]) / 1e3
                        except ValueError:
                            pass
                # wall minus the start-up run is the survey's method (and what the reference arm gets), but two index loads of ~15-30 s differ by
                # seconds; the command line's own clock around its mapping pass is exact but excludes the final junction collapse and the
                # tear-down.  The value reported is the SLOWER of the two.
                t_map = max(t_full - t_base, pass_wall or 0.0, 1e-3)
                cli = {"value": rp * rep / t_map, "stage_times_from_Log_out": host_lines, "mapping_pass_wall_s": pass_wall,
                       "pairs_per_s_by_wall_minus_startup": rp * rep / max(1e-3, t_full - t_base),
                       "pairs_per_s_by_mapping_pass_wall": (rp * rep / pass_wall) if pass_wall else None, "unit": UNIT, "pairs": rp * rep, "wall_s": t_full, "startup_and_index_load_s": t_base, "host_threads": threads, "cpus_allowed_by_cgroup": cpus_allowed,
                       "scope": "star_b200/bin/STAR: FASTQ files -> Aligned.out.sam + SJ.out.tab + Log.final.out, wall clock minus a --readMapNumber 1 run (same files and scope as the reference arm)"}
                # the command line's records for the sample equal the engine's input order: check them against the reference's on a small prefix
                try:
                    pn = min(rp, 20000)
                    q1, q2 = os.path.join(workdir, "par_1.fq"), os.path.join(workdir, "par_2.fq")
                    synth.write_fastq(m1[:pn], q1)
                    synth.write_fastq(m2[:pn], q2)
                    cli_run(idx, q1, q2, os.path.join(workdir, "cli_par"), threads, [], local_rank)
                    if os.path.exists(REF_STAR):
                        out_r = os.path.join(workdir, "ref_par")
                        shutil.rmtree(out_r, ignore_errors=True)
                        os.makedirs(out_r)
                        subprocess.check_call([REF_STAR, "--genomeDir", idx, "--readFilesIn", q1, q2, "--outFileNamePrefix", out_r + "/", "--runThreadN", "1"], stdout=subprocess.DEVNULL)
                        same_sam = sam_records(os.path.join(workdir, "cli_par", "Aligned.out.sam")) == sam_records(os.path.join(out_r, "Aligned.out.sam"))
                        same_sj = open(os.path.join(workdir, "cli_par", "SJ.out.tab"), "rb").read() == open(os.path.join(out_r, "SJ.out.tab"), "rb").read()
                        cli["parity_vs_reference"] = {"pairs": pn, "sam_records_equal": bool(same_sam), "sj_out_tab_equal": bool(same_sj),
                                                      "checker": "oracle/_ref/STAR --runThreadN 1 (unmodified reference), byte comparison"}
                        if not (same_sam and same_sj):
                            log("PARITY FAILURE: command-line output differs from the reference on the bench genome")
                            rc_exit = 3
                except subprocess.CalledProcessError as e:
                    cli["parity_vs_reference"] = {"error": str(e)}
                    rc_exit = 3
                for d in ("cli_base", "cli_run", "cli_par", "ref_par"):
                    shutil.rmtree(os.path.join(workdir, d), ignore_errors=True)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": t_val / a.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/int64",
                "data": "synthetic",
                "config": dict(config, l2_policy="inputs larger than L2 (index %.1f GB + reads %d MB per step, L2 126 MB)" % ((index.view.contents.nSAbyte + index.view.contents.nGenome + index.view.contents.nSAibyte) / 1e9, seq.nbytes >> 20),
                               parallelism="reads sharded across %d GPU(s), index replicated, one NCCL allreduce of the counters" % world,
                               mapped_fraction=float((res_np["unmapType"] < 0).mean()), overflow_tier_reads_per_step=int(last.slow_path_reads),
                               flat_path_reads_per_step=int(last.heavy_reads), flat_path_ms=float(last.ms_heavy), alignments_per_step=int(n_al),
                               stitch_nodes_per_pair=float(last.stitch_nodes) / n, sa_rows_enumerated_per_pair=float(last.sa_enumerated) / n,
                               wall_s_value_leg=wall, index_build=build, index_host_load_s=round(t_index_host, 1), engine_init_s=round(t_engine_init, 1)),
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "ms_per_step": wall_e2e / a.steps * 1e3,
                        "scope": "star_gpu_map_chunk (C-ABI) with pinned host buffers: packed sequences in, alignment records out"},
                "cli_e2e": cli, "parity_sample": parity,
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu}
        print(json.dumps(line), flush=True)
    if eng is not None:
        eng.close()
    index.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return rc_exit


if __name__ == "__main__":
    sys.exit(main())
