#!/usr/bin/env python3
"""bench.py -- k-mer insert+lookup throughput of the B200 engine on BASELINE.json config 2.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): 10 M synthetic 150 bp SE reads from a 100 Mbp random genome, 0.5 % substitutions, `-gs 100`
k-mer lengths (prefix 12, p17/s20/b24), original order.  The job is ONE stream of reads (fqsqueezer_b200/synth.py: job_chunk) cut
into reads_blocks exactly where the reference cuts the corresponding FASTQ (16 MiB slabs, reads_block.h:121-169 -> 196 blocks) and
every block into calc_no_synchronizations(g) + 1 sync segments (application.h:85-92); every segment is one fqsk_segment + fqsk_sync.

A STEP is 1/K of that job: step j covers blocks [196 j / K, 196 (j + 1) / K) (1 <= K <= 196), so any --steps spans both regimes of the job -- the
EARLY one (blocks 0..99: 100 - g sync segments per block, latency bound) and the STEADY one (blocks 100+: one 51 k-read segment per
block) -- which are also timed and reported separately (`regimes`).  The W warm-up steps run the first W steps of the job on a
throw-away engine (same work, untimed).

value  : bases/s with the reads already resident in HBM (fqsk_segment_device), timed with CUDA events on the engine's stream.
e2e    : the same steps through the host-buffer C-ABI calls (fqsk_submit_ctx / fqsk_collect per sync segment): H2D of the reads and D2H of every per-base
         record inside the timed region.
parity_check : device-side checksums (fqsk_recs_checksum) of every sync segment of the first blocks of the timed job against the
         REAL reference's records for the same reads (tests/golden/bench_config2_ref_checksums.npz, produced once by
         oracle/make_bench_golden.py from the tapped fqs-1.1 at -t 1).
--dump-outputs DIR : after the timed steps, what fqsk_segment_device handed its caller in every sync segment of the LAST timed step, as
         float64 .npy files: the number of records and their device checksum per segment, and a fixed, seeded sample of the per-base
         records (at most 2^19 + one per segment, under 40 MB in all).  The inputs depend on nothing but the arguments, so two builds
         can be compared output for output.  Taking the sample waits for every segment of that step inside the timed region, so the
         line then carries "timing_comparable": false.  Not with --impl reference or N > 1.
N > 1  : ONE job over N GPUs, tables hash-sharded by the reference's owner keys (reference `-t N` semantics; scaling "strong");
         `--replicas` runs N independent engines instead (weak scaling, no exchange).
roofline / cpu_baseline / compress_e2e: see DESIGN.md section 7.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from fqsqueezer_b200 import schedule as S  # noqa: E402
from fqsqueezer_b200 import synth  # noqa: E402

METRIC = "kmer_insert_lookup_bases_per_s"
UNIT = "bases/s"
L = 150
GENOME = 100_000_000
SEED = 43
GS = 100
JOB_READS = 10_000_000
RESERVE_READS = 52_000              # largest reads_block of the job (51 694 reads: the first one, short ids)
B_ALG = 251.5                       # algorithmic bytes per base, SURVEY.md section 8d (config 2)
EARLY_BLOCKS = 100                  # blocks 0..99 have intra-block syncs (application.h:85-92)
PHASE_ALG = {"lookup": 127 * 32 / 150.0, "sync_apply": (127 + 131) * 64 / 150.0, "sync_siv": 134 * 128 / 150.0}
PHASE_KERNEL = {"prep": "k_prep", "lookup": "k_lookup", "partial": "k_partial", "walk": "k_walk", "compact": "k_compact2+scans",
                "sort": "k_delta_build / row grouping", "local": "k_local", "rough": "k_rough", "fold": "k_fold", "sync_locate": "k_locate_heads / k_sync_rank",
                "sync_apply": "k_apply_keys / k_sync_apply / k_insert_fast", "sync_siv": "k_siv_increment", "mt": "k_mt_extend"}
GOLDEN_SUMS = os.path.join(ROOT, "tests", "golden", "bench_config2_ref_checksums.npz")


def job_blocks():
    """Read ranges [first, last) of the job's reads_blocks, cut where the reference cuts the FASTQ (reads_block.h:121-169)."""
    return S.split_blocks(synth.fastq_record_sizes(1, JOB_READS, L))


def workload_config(n_gpus, replicas=False):
    """Identical for both arms (`--impl reference` prints the same dict): what is measured, not how."""
    c = {"workload": "BASELINE config 2: 10 M 150bp SE reads, 100 Mbp random genome, 0.5% subs, -gs 100 (p17/s20/b24), -om o; the whole job, reads_blocks and sync schedule as the reference cuts them",
         "job_reads": JOB_READS, "job_blocks": 196, "read_len": L, "step": "1/K of the job's blocks",
         "l2": "tables (4 GiB p-mer array + GiB-scale b/s tables) are far larger than L2; no flush needed"}
    if n_gpus > 1:
        c["parallelism"] = (f"{n_gpus} independent replicas" if replicas else
                            f"ONE job over {n_gpus} GPUs: every reads_block split among {n_gpus} workers, tables hash-sharded by the reference's owner keys (fqs-1.1 -t {n_gpus} semantics)")
    return c


class JobReads:
    """The job's read stream, generated chunk by chunk (deterministic in the chunk number) and served block by block."""

    def __init__(self, genome):
        self.genome, self.chunks = genome, {}

    def _chunk(self, c):
        if c not in self.chunks:
            self.chunks[c] = synth.job_chunk(self.genome, c, L)[0]
            for k in [k for k in self.chunks if k < c - 2]:
                del self.chunks[k]
        return self.chunks[c]

    def codes(self, first, last):
        parts = []
        a = first
        while a < last:
            c = a // synth.JOB_CHUNK
            lo = a - c * synth.JOB_CHUNK
            hi = min(synth.JOB_CHUNK, lo + (last - a))
            parts.append(self._chunk(c)[lo:hi])
            a += hi - lo
        return parts[0] if len(parts) == 1 else np.concatenate(parts)


def codes_to_slab(codes):
    """DNA lines only ('ACGT...\\n'): ids and qualities never reach the k-mer path."""
    n = codes.shape[0]
    slab = np.empty((n, L + 1), np.uint8)
    slab[:, :L] = synth.codes_to_ascii(codes)
    slab[:, L] = 10
    off = (np.arange(n, dtype=np.uint64) * np.uint64(L + 1))
    ln = np.full(n, L, np.uint32)
    return slab.reshape(-1), off, ln


DUMP_SAMPLE = 1 << 19               # records of the last timed step kept by --dump-outputs (8 float64 columns each: 32 MiB)
DUMP_SEED = 7
REC_FIELDS = ["pos", "c0", "c1", "c2", "c3", "cor_pos", "level", "rough"]      # fqsk_base_rec (include/fqsk.h) without its padding


class _DeviceBytes:
    """A device buffer owned by the engine, handed to torch without a copy (__cuda_array_interface__)."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3}


class LastStepOutputs:
    """--dump-outputs: per sync segment of the last timed step, the records fqsk_segment_device leaves in device memory for its caller --
    their number, the device checksum of all of them (fqsk_recs_checksum) and a seeded sample of them; the sample takes a share of
    DUMP_SAMPLE proportional to the segment's reads, at positions drawn from a generator seeded with the segment's ordinal."""

    def __init__(self, reads_in_step, dev):
        self.reads_in_step, self.dev = reads_in_step, dev
        self.n_recs, self.sums, self.index, self.rows = [], [], [], []
        self.first = 0                  # position of the current segment's first record in the step's record stream

    def capture(self, eng, n_reads):
        import torch
        from fqsqueezer_b200 import engine as E
        cs, n = eng.recs_checksum()     # settles the segment and waits for the engine's stream
        ptr, n_dev = eng.device_recs()
        assert n_dev == n, (n_dev, n)
        m = min(n, -(-DUMP_SAMPLE * n_reads // self.reads_in_step))
        idx = np.unique(np.random.default_rng([DUMP_SEED, len(self.n_recs)]).integers(0, n, m)) if m else np.zeros(0, np.int64)
        if len(idx):
            rb = E.REC_DTYPE.itemsize
            recs = torch.as_tensor(_DeviceBytes(ptr, n * rb), device=self.dev).view(torch.int32).view(n, rb // 4)
            w = recs[torch.from_numpy(idx).to(self.dev)].cpu().numpy().view(np.uint32)      # .cpu() waits: the next segment reuses the buffer
            self.rows.append(np.stack([w[:, 0], w[:, 1], w[:, 2], w[:, 3], w[:, 4], w[:, 5], w[:, 6] & 0xFF, (w[:, 6] >> 8) & 0xFF], axis=1).astype(np.float64))
            self.index.append((self.first + idx).astype(np.float64))
        self.n_recs.append(n)
        self.sums.append((cs >> 32, cs & 0xFFFFFFFF))
        self.first += n

    def write(self, out_dir):
        os.makedirs(out_dir, exist_ok=True)
        arrays = {"segment_n_records": np.array(self.n_recs, np.float64),
                  "segment_checksum_hi_lo": np.array(self.sums, np.float64).reshape(-1, 2),
                  "records_sample": np.concatenate(self.rows) if self.rows else np.zeros((0, len(REC_FIELDS)), np.float64),
                  "records_sample_index": np.concatenate(self.index) if self.index else np.zeros(0, np.float64)}
        for name, a in arrays.items():
            np.save(os.path.join(out_dir, name + ".npy"), a)
        return {"dir": out_dir, "segments": len(self.n_recs), "records": int(self.first), "sampled": len(arrays["records_sample_index"]),
                "records_sample_columns": REC_FIELDS, "bytes": sum(a.nbytes for a in arrays.values())}


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons DURING the timed region.  NVML in-process (nvidia_ml_py): a query costs microseconds and does not touch
    the CUDA context; spawning nvidia-smi five times a second next to a job that launches 60 000 kernels a second did (fork + NVML init per sample)."""

    def __init__(self, index, hz=2.0):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows, self.hz, self.mx = index, False, [], hz, None
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            uuid = None
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(index).uuid)
            except Exception:
                pass
            self.dev = None
            if uuid:
                for i in range(pynvml.nvmlDeviceGetCount()):
                    hnd = pynvml.nvmlDeviceGetHandleByIndex(i)
                    u = pynvml.nvmlDeviceGetUUID(hnd)
                    u = u.decode() if isinstance(u, bytes) else u
                    if uuid in u or u.replace("GPU-", "") == uuid:
                        self.dev = hnd
            if self.dev is None:
                self.dev = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.dev, n.NVML_CLOCK_SM)
        if self.mx is None:
            self.mx = n.nvmlDeviceGetMaxClockInfo(self.dev, n.NVML_CLOCK_SM)
        mx = self.mx
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(self.dev)
        except Exception:
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.dev)
        act = lambda bit: "Active" if (r & bit) else "Not Active"
        return [str(sm), str(mx), "0", act(n.nvmlClocksThrottleReasonHwSlowdown), act(n.nvmlClocksThrottleReasonHwThermalSlowdown),
                act(n.nvmlClocksThrottleReasonSwThermalSlowdown), act(n.nvmlClocksThrottleReasonSwPowerCap)]

    def run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    self.rows.append(self._sample_nvml())
                else:
                    out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                         capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(1.0 / self.hz if self.nvml is not None else 0.5)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        mx = max(float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows if len(r) > 3 + i)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons, "samples": len(self.rows), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic():
    """DRAM bytes of one steady-state step from the committed ncu capture of this round (profiles/r02_traffic.json), or None."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            pass
    return None


# ------------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the unmodified fqs-1.1 compiled from /root/reference (oracle/_ref/fqs-1.1)
# ------------------------------------------------------------------------------------------------------------------
def run_reference(reads: JobReads, n_reads, threads):
    """Times the unmodified fqs-1.1 on the FIRST n_reads reads of the job (the same reads, ids and block cuts the GPU arm starts with).
    Its 'Processing time' starts with the construction of the CPU tables (4 GiB p-mer array + 5 M sub-tables at -gs 100: seconds,
    independent of the input), which the 10 M-read job amortises and a bounded sample does not: the same binary is therefore also
    timed on an 8-read file and that start-up is reported and taken off -- as the GPU arm's table construction (fqsk_create) lies
    outside its timed region too."""
    from oracle import oracle as O          # checker side only: this function never touches the product path
    if not os.path.exists(O.REF_BIN):
        return None

    def one(codes, tmp, name):
        fq = os.path.join(tmp, name + ".fastq")
        nbytes = synth.write_fastq(fq, codes, np.zeros(codes.shape, bool), seed=1)
        cmd = [O.REF_BIN, "e", "-s", "-om", "o", "-qm", "o", "-im", "o", "-gs", str(GS), "-t", str(threads), "-v", "0", "-out", os.path.join(tmp, name + ".fqs"), fq]
        t = time.time()
        r = subprocess.run(cmd, capture_output=True, text=True, cwd=tmp)
        wall = time.time() - t
        m = re.search(r"Processing time:\s*([0-9.eE+-]+)", r.stdout + r.stderr)
        return (float(m.group(1)) if m else wall), nbytes

    codes = reads.codes(0, n_reads)
    with tempfile.TemporaryDirectory() as tmp:
        startup, _ = one(codes[:8], tmp, "tiny")
        secs, nbytes = one(codes, tmp, "s")
    net = max(secs - startup, 0.05 * secs)
    return {"bases": n_reads * L, "seconds": net, "seconds_total": secs, "startup_seconds": startup, "fastq_bytes": nbytes}


def run_compress_e2e(reads: JobReads, n_reads):
    """BASELINE.json's second metric, `e2e compress MB/s`: the reference compressor with its k-mer engine bound to libfqsk.so
    (host/_bin/fqs-1.1-fqsk: host/build_host.py + host/fqsk_live.h, the integration of INTEGRATION.md) against the unmodified
    fqs-1.1 at -t 1 -- the parity configuration -- on the same FASTQ (the first n_reads reads of the job): FASTQ bytes / seconds,
    and whether the two .fqs files are byte-identical.  Everything outside the k-mer engine is the reference's own host code."""
    from oracle import oracle as O          # only to locate the unmodified reference binary (the baseline of this leg)
    live = os.path.join(ROOT, "host", "_bin", "fqs-1.1-fqsk")
    lib = os.path.join(ROOT, "fqsqueezer_b200", "libfqsk.so")
    if not (os.path.exists(live) and os.path.exists(O.REF_BIN)):
        return {"unavailable": "host/_bin/fqs-1.1-fqsk or oracle/_ref/fqs-1.1 not built"}
    codes = reads.codes(0, n_reads)
    rng = np.random.default_rng(4242)
    err = rng.random(codes.shape) < 0.005          # only decides where the '#' qualities sit
    with tempfile.TemporaryDirectory() as tmp:
        fq = os.path.join(tmp, "s.fastq")
        nbytes = synth.write_fastq(fq, codes, err, seed=1)
        base = ["e", "-s", "-om", "o", "-qm", "o", "-im", "o", "-gs", str(GS), "-t", "1", "-v", "0"]

        def one(exe, out, env=None, files=None):
            t = time.time()
            r = subprocess.run([exe, *base, "-out", out, *(files or [fq])], capture_output=True, text=True, cwd=tmp, env=env, timeout=600)
            wall = time.time() - t
            if r.returncode != 0:
                raise RuntimeError(f"{os.path.basename(exe)} exit {r.returncode}: {r.stderr[-300:]}")
            m = re.search(r"Processing time:\s*([0-9.eE+-]+)", r.stdout + r.stderr)
            return (float(m.group(1)) if m else wall), wall, r.stderr

        env = dict(os.environ, FQSK_LIB=lib, FQSK_VERBOSE="1")
        one(live, os.path.join(tmp, "w.fqs"), env)                     # warm-up: CUDA context, module load, page cache
        t_live, wall_live, log = one(live, os.path.join(tmp, "a.fqs"), env)
        t_ref, wall_ref, _ = one(O.REF_BIN, os.path.join(tmp, "b.fqs"))
        # start-up of either binary (table construction: fqsk_create = CUDA context + 12 GiB of HBM tables; reference = its CPU tables)
        # on an 8-read file, reported beside the totals
        tiny = os.path.join(tmp, "tiny.fastq")
        synth.write_fastq(tiny, codes[:8], err[:8], seed=1)
        s_live, _, _ = one(live, os.path.join(tmp, "t1.fqs"), env, [tiny])
        s_ref, _, _ = one(O.REF_BIN, os.path.join(tmp, "t2.fqs"), None, [tiny])
        same = open(os.path.join(tmp, "a.fqs"), "rb").read() == open(os.path.join(tmp, "b.fqs"), "rb").read()
        fqs_bytes = os.path.getsize(os.path.join(tmp, "a.fqs"))
    m = re.search(r"([0-9.]+) s inside the engine calls, (\d+) kernel launches", log)
    mw = re.search(r"([0-9.]+) s waiting for the engine", log)
    return {"value": nbytes / 1e6 / t_live, "unit": "MB/s", "reference_t1": nbytes / 1e6 / t_ref, "speedup_vs_t1": t_ref / t_live,
            "byte_identical": bool(same), "fastq_bytes": nbytes, "fqs_bytes": fqs_bytes, "seconds": t_live, "reference_seconds": t_ref,
            "startup_seconds": s_live, "reference_startup_seconds": s_ref,
            "value_without_startup": nbytes / 1e6 / max(t_live - s_live, 1e-3), "reference_t1_without_startup": nbytes / 1e6 / max(t_ref - s_ref, 1e-3),
            "engine_call_seconds": float(m.group(1)) if m else None, "engine_wait_seconds": float(mw.group(1)) if mw else None, "gpu_launches": int(m.group(2)) if m else None,
            "sample": f"the first {n_reads} reads of the job ({nbytes / 1e6:.1f} MB FASTQ), e -s -om o -qm o -im o -gs {GS} -t 1: fqs-1.1-fqsk (reference host code, k-mer engine on the GPU through the C-ABI) vs the unmodified fqs-1.1; 'Processing time' of each, start-up included; the start-up of each binary (same options, 8-read file) is reported separately"}


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = min(os.cpu_count() or 1, 64)
    reads = JobReads(synth.make_genome(GENOME, SEED))
    per_step = max(200, args.ref_sample_reads // max(args.steps, 1))     # K steps of a bounded sample of the job's first reads
    if args.warmup:
        run_reference(reads, min(per_step * args.warmup, 10_000), threads)
    res = run_reference(reads, per_step * args.steps, threads)
    if res is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/fqs-1.1 not built"}))
        return 0
    t1 = run_reference(reads, args.ref_t1_reads, 1) if args.ref_t1_reads else None
    v = res["bases"] / res["seconds"]
    sample = (f"the first {per_step * args.steps} reads of the job ({args.steps} steps x {per_step}; the reads the GPU arm starts with), fqs-1.1 e -s -om o -qm o -im o -gs {GS} -t {threads}: "
              f"'Processing time' {res['seconds_total']:.2f} s minus {res['startup_seconds']:.2f} s of table construction (same binary on an 8-read file); whole compressor")
    cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "reference", "sample": sample}
    if t1:
        cpu["t1_value"] = t1["bases"] / t1["seconds"]
        cpu["t1_sample"] = f"-t 1 on the first {args.ref_t1_reads} reads: {t1['seconds_total']:.2f} s minus {t1['startup_seconds']:.2f} s of table construction"
    line = {"metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * res["seconds"] / args.steps, "higher_is_better": True, "scaling": "strong" if args.gpus > 1 and not args.replicas else "weak", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic", "impl": "reference", "config": workload_config(args.gpus, args.replicas),
            "cpu_baseline": cpu,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------------------------
# parity check: device-side checksums of the first blocks' segments against the real reference's records
# ------------------------------------------------------------------------------------------------------------------
def parity_check(make_engine, reads: JobReads, blocks, max_blocks, dev):
    import torch
    if not os.path.exists(GOLDEN_SUMS):
        return {"ok": None, "unavailable": "tests/golden/bench_config2_ref_checksums.npz missing"}
    z = np.load(GOLDEN_SUMS)
    nb = min(int(len(z["segs_per_block"])), max_blocks, len(blocks))
    if (int(z["gs"]), int(z["genome"]), int(z["seed"]), int(z["read_len"])) != (GS, GENOME, SEED, L):
        return {"ok": None, "unavailable": "golden checksums belong to another workload"}
    eng = make_engine()
    seg, n_rec, bad = 0, 0, []
    t0 = time.time()
    for g in range(nb):
        f, l = blocks[g]
        if (int(z["block_first"][g]), int(z["block_last"][g])) != (f, l):
            return {"ok": False, "error": f"block {g} is reads [{f}, {l}) here, [{int(z['block_first'][g])}, {int(z['block_last'][g])}) in the reference run"}
        codes = reads.codes(f, l)
        t = torch.from_numpy(synth.codes_to_ascii(codes).reshape(-1)).to(dev)
        d_off = torch.arange(l - f, dtype=torch.int64, device=dev) * L
        d_len = torch.full((l - f,), L, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()      # the engine works on its own non-blocking stream: torch's copies / fills must have landed before it reads them
        sched = list(S.segments(0, l - f, S.calc_no_synchronizations(g, l - f, 1)))
        if len(sched) != int(z["segs_per_block"][g]):
            return {"ok": False, "error": f"block {g}: {len(sched)} segments here, {int(z['segs_per_block'][g])} in the reference run"}
        eng.block_start()
        for a, b in sched:
            eng.segment_device(t.data_ptr() + a * L, (b - a) * L, d_off.data_ptr(), d_len.data_ptr(), b - a, want_n_recs=False)
            cs, n = eng.recs_checksum()
            if n != int(z["seg_nrecs"][seg]) or cs != int(z["seg_sum"][seg]):
                bad.append(seg)
            n_rec += n
            seg += 1
            eng.sync()
    eng.close()
    return {"ok": len(bad) == 0, "blocks": nb, "segments": seg, "records": n_rec, "mismatching_segments": bad[:8], "seconds": round(time.time() - t0, 2),
            "checker": "per-segment record checksums of the REAL reference (tapped fqs-1.1 -t 1 on the same reads, oracle/make_bench_golden.py) vs fqsk_recs_checksum on the device"}


# ------------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-per-segment", action="store_true", help="e2e leg: one fqsk_submit_ctx / fqsk_collect call per sync segment from Python instead of one fqsk_block_stream call per reads_block")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--clock-hz", type=float, default=2.0, help="NVML samples per second of SM clock + throttle reasons during the timed region (0: one sample before and one after it)")
    ap.add_argument("--short-warmup", action="store_true", help="warm up with the first W steps only (default: W steps, then the rest of the job, all on a throw-away engine)")
    ap.add_argument("--replicas", action="store_true", help="N > 1: N independent engines (weak scaling) instead of ONE job over hash-sharded tables")
    ap.add_argument("--shard", action="store_true", help="(default at N > 1; kept for compatibility)")
    ap.add_argument("--no-phase-events", action="store_true", help="skip the second pass that brackets the internal phases with CUDA events")
    ap.add_argument("--no-parity-check", action="store_true")
    ap.add_argument("--parity-blocks", type=int, default=8, help="blocks of the job checked against the reference's golden checksums")
    ap.add_argument("--ref-sample-reads", type=int, default=120_000, help="bounded sample of the reference legs (-t nproc)")
    ap.add_argument("--ref-t1-reads", type=int, default=16_000, help="bounded sample of the reference's -t 1 figure (0 = skip)")
    ap.add_argument("--no-compress-e2e", action="store_true", help="skip the whole-compressor leg (fqs-1.1-fqsk vs fqs-1.1 -t 1)")
    ap.add_argument("--compress-sample-reads", type=int, default=60_000)
    ap.add_argument("--max-blocks", type=int, default=0, help="debug: stop the job after this many blocks")
    ap.add_argument("--trace-blocks", type=int, default=0, help="print per-block phase ms every N blocks to stderr")
    ap.add_argument("--profile-block", type=int, default=-1, help="cudaProfilerStart/Stop around this block (for ncu --profile-from-start off)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the records of the last timed step (per-segment counts and checksums, "
                    "a seeded sample of the records) as DIR/<name>.npy; one engine only")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs: the records come from the engine's timed path; --impl reference has none")
        return reference_arm(args)

    import torch
    from fqsqueezer_b200 import engine as E

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the k-mer path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    sharded = world > 1 and not args.replicas

    pref, p, s, b = E.kmer_params(GS)
    reads = JobReads(synth.make_genome(GENOME, SEED))
    blocks = job_blocks()
    if args.max_blocks:
        blocks = blocks[: args.max_blocks]
    NB = len(blocks)
    K = args.steps
    if not 1 <= K <= NB:
        raise SystemExit(f"--steps {K}: a step is 1/K of the job's {NB} reads_blocks, so 1 <= --steps <= {NB}")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs: one engine only (no --gpus > 1)")
    step_of_block = [g * K // NB for g in range(NB)]
    # warm-up: W steps of the job on a throw-away engine -- and, unless --short-warmup, the rest of the job behind them: a fresh box needs
    # seconds, not steps, until its host side runs at speed (the first bench run on a fresh box measured 3x the launch work of the second,
    # profiles/r02_bench_first_run_on_a_fresh_box.json), and the later blocks use launch paths (51 000-read segments) the first W steps never touch
    warm_blocks = [g for g in range(NB) if step_of_block[g] < args.warmup or not args.short_warmup]
    n_early = min(EARLY_BLOCKS, NB)

    # this rank's share of every block: everything (1 GPU / replicas) or worker `rank`'s slice (sharded: PartitionForWorkers)
    def my_segments(g):
        f, l = blocks[g]
        if sharded:
            return S.worker_segments(0, l - f, g, world, rank)
        return list(S.segments(0, l - f, S.calc_no_synchronizations(g, l - f, 1)))

    sched = [my_segments(g) for g in range(NB)]
    if sharded:
        from fqsqueezer_b200 import sharded as SH

    def make_engine(profile=False, e2e=False):
        rr, rb = RESERVE_READS, RESERVE_READS * (L + (1 if e2e else 0))
        if sharded:
            return SH.ShardedKmerEngine(p, s, b, pref, rank, world, device=local_rank, dist=dist, expected_kmers=(1 << 29) // world,
                                        reserve_reads=rr // world + 16, reserve_bytes=(rr // world + 16) * (L + 1), profile=profile)
        return E.KmerEngine(p, s, b, pref, device=local_rank, expected_kmers=1 << 29, profile=profile, reserve_reads=rr, reserve_bytes=rb)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- value: reads resident in HBM ----------------
    t_create = time.time()
    eng = make_engine(profile=bool(args.trace_blocks))
    torch.cuda.synchronize()
    create_s = time.time() - t_create
    d_off = torch.arange(RESERVE_READS + 16, dtype=torch.int64, device=dev) * L      # same offsets for every block (relative to the segment's first read)
    d_len = torch.full((RESERVE_READS + 16,), L, dtype=torch.int32, device=dev)
    d_blocks = []
    for g in range(NB):
        f, l = blocks[g]
        lo, hi = sched[g][0][0], sched[g][-1][1]
        codes = reads.codes(f + lo, f + hi) if (replica_shift := 0) == 0 else None
        d_blocks.append((lo, torch.from_numpy(synth.codes_to_ascii(codes).reshape(-1)).to(dev)))
    torch.cuda.synchronize()

    def run_block_device(g, e, capture=None):
        e.block_start()
        lo, t = d_blocks[g]
        base = t.data_ptr()
        segs = sched[g]
        for k, (a, bb) in enumerate(segs):
            n = bb - a
            e.segment_device(base + (a - lo) * L, n * L, d_off.data_ptr(), d_len.data_ptr(), n, want_n_recs=False)
            if capture is not None:
                capture(e, n)
            if k + 1 < len(segs):      # the worker loop knows its next segment (application.cpp:617-662): its read-only preparation runs ahead
                a2, b2 = segs[k + 1]
                e.announce_device(base + (a2 - lo) * L, (b2 - a2) * L, d_off.data_ptr(), d_len.data_ptr(), b2 - a2)
            e.sync()

    # warm-up: the first W steps of the job on a throw-away engine (a fresh box starts with idle clocks and a cold driver)
    scratch = make_engine()
    for g in warm_blocks:
        run_block_device(g, scratch)
    scratch.close()
    del scratch
    st0 = eng.stats()
    sampler = ClockSampler(local_rank, hz=args.clock_hz or 2.0)
    if args.clock_hz > 0:
        sampler.start()
    elif sampler.nvml is not None:
        sampler.rows.append(sampler._sample_nvml())
    barrier()
    t_wall = time.time()
    prev_prof, t_prev = eng.profile(), time.time()
    regime_ms = {"early": 0.0, "steady": 0.0}
    seg_early = 0
    last_step = None
    if args.dump_outputs:
        last_step = LastStepOutputs(sum(sched[g][-1][1] - sched[g][0][0] for g in range(NB) if step_of_block[g] == K - 1), dev)

    def run_range(g0, g1, key):
        nonlocal prev_prof, t_prev
        if g0 >= g1:
            return
        eng.timer_begin()
        for g in range(g0, g1):
            if g == args.profile_block:
                torch.cuda.cudart().cudaProfilerStart()
            run_block_device(g, eng, last_step.capture if last_step is not None and step_of_block[g] == K - 1 else None)
            if g == args.profile_block:
                torch.cuda.cudart().cudaProfilerStop()
            if args.trace_blocks and (g % args.trace_blocks == 0 or g == NB - 1):
                pr = eng.profile()
                print(f"block {g} ({len(sched[g])} segments): wall {1e3 * (time.time() - t_prev):.1f} ms " +
                      str({k: round(pr[k] - prev_prof[k], 2) for k in pr}) + " " +
                      str({k: v for k, v in eng.stats().items() if k in ("n_hot_segments", "n_replays", "bmer_buckets", "smer_buckets", "bmer_stash_used", "n_bmers", "n_smers", "draws_b")}),
                      file=sys.stderr, flush=True)
            if args.trace_blocks:
                prev_prof, t_prev = eng.profile(), time.time()
        regime_ms[key] += eng.timer_end()

    run_range(0, n_early, "early")
    seg_early = eng.stats()["n_segments"] - st0["n_segments"]
    run_range(n_early, NB, "steady")
    barrier()
    wall_ms = (time.time() - t_wall) * 1e3
    sampler.stop_flag = True
    if args.clock_hz <= 0 and sampler.nvml is not None:
        sampler.rows.append(sampler._sample_nvml())
    st1 = eng.stats()
    dev_ms = regime_ms["early"] + regime_ms["steady"]
    ms = torch.tensor([dev_ms, regime_ms["early"], regime_ms["steady"]], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    dev_ms_max, early_ms, steady_ms = (float(x) for x in ms.tolist())
    job_bases = sum(l - f for f, l in blocks) * L
    early_bases = sum(l - f for f, l in blocks[:n_early]) * L
    total_bases = job_bases * (world if (world > 1 and not sharded) else 1)       # replicas: every rank runs the whole job
    value = total_bases / (dev_ms_max / 1e3)
    n_seg = st1["n_segments"] - st0["n_segments"]
    launches = st1["kernel_launches"] - st0["kernel_launches"]
    if dist is not None:
        lt = torch.tensor([launches], dtype=torch.int64, device=dev)
        dist.all_reduce(lt)
        launches = int(lt.item())
    eng.close()
    dumped = last_step.write(args.dump_outputs) if last_step is not None else None

    # ---------------- phase shares: the same pass again with CUDA-event brackets around the internal phases ----------------
    phases = None
    if not args.no_phase_events and not sharded:
        engp = make_engine(profile=True)
        prof0 = engp.profile()
        for g in range(NB):
            run_block_device(g, engp)
        prof1 = engp.profile()
        phases = {k: prof1[k] - prof0[k] for k in prof1}
        engp.close()
    del d_blocks
    torch.cuda.empty_cache()

    # ---------------- parity: device-side checksums of the first blocks against the real reference ----------------
    parity = None
    if not args.no_parity_check and not sharded and rank == 0:
        parity = parity_check(make_engine, reads, blocks, args.parity_blocks, dev)

    # ---------------- e2e: host buffers through fqsk_submit / fqsk_collect ----------------
    e2e = None
    if not args.no_e2e and not sharded:
        eng2 = make_engine(e2e=True)
        slabs = [codes_to_slab(reads.codes(*blocks[g])) for g in range(NB)]

        seg_ends = [np.array([bb for _, bb in sched[g]], np.uint32) for g in range(NB)]

        def run_block_host(g, pend, e):
            """One reads_block through fqsk_block_stream (fqsk_submit_ctx / fqsk_collect per sync segment, two segments in flight: segment
            n + 1 is submitted before n is collected -- the point where the reference's host-side coder consumes the records of n;
            host/fqsk_live.h makes the same calls one by one).  The pipeline runs across block boundaries: the block's last segment stays in
            flight and is collected by the next call -- the records of a 51 000-read segment take as long to reach the host as the next one
            takes to compute.  --e2e-per-segment: the same calls made one by one from Python (5 146 x 2 ctypes calls)."""
            slab, off, ln = slabs[g]
            nb = 0
            if not args.e2e_per_segment:
                for recs in e.block_stream(slab, off, ln, seg_ends[g], ctx=True):
                    nb += recs.nbytes
                return nb + len(off), None
            e.block_start()
            for a, bb in sched[g]:
                t = e.submit(slab, off[a:bb], ln[a:bb], ctx=True)
                if pend is not None:
                    recs, dup, _ = e.collect(pend)
                    nb += recs.nbytes + dup.nbytes
                pend = t
            return nb, pend

        def drain(pend, e):
            if not args.e2e_per_segment:
                recs = e.stream_finish()
                return recs.nbytes if recs is not None else 0
            if pend is None:
                return 0
            recs, dup, _ = e.collect(pend)
            return recs.nbytes + dup.nbytes

        scratch = make_engine(e2e=True)
        pend = None
        for g in warm_blocks:
            _, pend = run_block_host(g, pend, scratch)
        drain(pend, scratch)
        pend = None
        scratch.close()
        barrier()
        t0 = time.time()
        d2h = 0
        for g in range(NB):
            nb, pend = run_block_host(g, pend, eng2)
            d2h += nb
        d2h += drain(pend, eng2)
        barrier()
        e2e_s = time.time() - t0
        st_e2e = eng2.stats()
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e = {"value": total_bases / float(t.item()), "unit": UNIT,
               "h2d_bytes_per_step": (JOB_READS if not args.max_blocks else blocks[-1][1]) * (L + 12) // K, "d2h_bytes_per_step": d2h // K,
               "host": {"api_ms": round(st_e2e["api_ns"] / 1e6, 1), "waiting_for_the_gpu_ms": round(st_e2e["look_wait_ns"] / 1e6, 1)},
               "call": "fqsk_submit_ctx + fqsk_collect per sync segment from Python" if args.e2e_per_segment else "fqsk_block_stream per reads_block (fqsk_submit_ctx + fqsk_collect per sync segment inside the library)",
               "note": "fqsk_submit_ctx / fqsk_collect (what the compiled drop-in calls) with host slab + read descriptors (H2D inside), one 16-byte context record per coded base (the 7 context ids + rank the range coder consumes, built on the device) copied back into page-locked host memory on a second stream, two segments in flight, across block boundaries too; wall clock incl. ctypes/numpy host code"}
        eng2.close()
        del slabs

    # ---------------- e2e of the sharded job: host buffers through the blocking pair, per rank ----------------
    if not args.no_e2e and sharded:
        def sharded_e2e():
            """Every rank codes its slice of every reads_block from HOST buffers: fqsk_segment (H2D of the reads, the segment, D2H of the
            28-byte count records into page-locked memory) + the device-driven sync, per sync segment -- the calls host/fqsk_live.h makes at
            -t N (fqsk_submit is not available on a sharded engine, so nothing overlaps the copies).  Wall clock, max over the ranks."""
            eng2 = make_engine(e2e=True)
            mine = []
            for g in range(NB):
                f, _ = blocks[g]
                lo, hi = sched[g][0][0], sched[g][-1][1]
                mine.append(codes_to_slab(reads.codes(f + lo, f + hi)) + (lo,))

            def run(g, e):
                slab, off, ln, lo = mine[g]
                e.block_start()
                nb = 0
                for a, bb in sched[g]:
                    recs, dup = e.segment(slab, off[a - lo:bb - lo], ln[a - lo:bb - lo], pinned=True)
                    nb += recs.nbytes + dup.nbytes
                    e.sync()
                return nb

            scratch = make_engine(e2e=True)
            for g in range(NB):
                if step_of_block[g] < args.warmup:
                    run(g, scratch)
            scratch.close()
            barrier()
            t0 = time.time()
            d2h = 0
            for g in range(NB):
                d2h += run(g, eng2)
            barrier()
            secs = time.time() - t0
            st_e2e = eng2.stats()
            eng2.close()
            t = torch.tensor([secs], dtype=torch.float64, device=dev)
            nbt = torch.tensor([d2h], dtype=torch.int64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(nbt)
            return {"value": total_bases / float(t.item()), "unit": UNIT,
                    "h2d_bytes_per_step": (JOB_READS if not args.max_blocks else blocks[-1][1]) * (L + 12) // K, "d2h_bytes_per_step": int(nbt.item()) // K,
                    "host": {"api_ms": round(st_e2e["api_ns"] / 1e6, 1), "waiting_for_the_gpu_ms": round(st_e2e["look_wait_ns"] / 1e6, 1)},
                    "call": "fqsk_segment + fqsk_sync_device per sync segment on every rank (blocking)",
                    "note": "ONE job over the ranks with host slabs: per sync segment H2D of the rank's reads, the segment, D2H of one 28-byte count record per coded base into page-locked memory, then the device-driven sync; h2d / d2h bytes are summed over the ranks; wall clock incl. ctypes/numpy host code, max over the ranks"}
        try:
            e2e = sharded_e2e()
        except Exception as ex:      # the device-timed line above stands on its own
            e2e = {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    # ---------------- roofline ----------------
    peak, peak_src = measured_peak()
    n_dev = world if sharded else 1
    step_achieved = B_ALG * job_bases / (dev_ms_max / 1e3) / 1e9
    traffic = measured_traffic()
    roof = {"bound": "hbm", "achieved": step_achieved, "peak": peak * n_dev, "unit": "GB/s", "frac": step_achieved / (peak * n_dev),
            "traffic": traffic.get("dram_bytes_per_steady_step") if traffic else None,
            "peak_source": peak_src,
            "kernel": "whole step (all kernels of fqsk_segment + fqsk_sync), 251.5 algorithmic B/base",
            "traffic_note": (traffic.get("note") if traffic else "no ncu capture of this round committed yet")}
    regimes = {}
    for key, ms_r, bases_r, blk, segs in (("early", early_ms, early_bases, f"0..{n_early - 1}", seg_early), ("steady", steady_ms, job_bases - early_bases, f"{n_early}..{NB - 1}", n_seg - seg_early)):
        if ms_r > 0:
            a = B_ALG * bases_r / (ms_r / 1e3) / 1e9
            regimes[key] = {"blocks": blk, "segments": int(segs), "ms": round(ms_r, 2), "ms_per_block": round(ms_r / max(1, (n_early if key == "early" else NB - n_early)), 3),
                            "bases_per_s": bases_r / (ms_r / 1e3), "achieved_GBps": a, "frac": a / (peak * n_dev)}
    if phases:
        dom = max(phases, key=lambda k: phases[k])
        dom_share = phases[dom] / max(sum(phases.values()), 1e-9)
        dom_alg = PHASE_ALG.get(dom, 0.0) * job_bases
        roof["dominant_kernel"] = {"name": PHASE_KERNEL.get(dom, dom), "share_of_device_time": dom_share, "ms_per_step": phases[dom] / K,
                                   "algorithmic_GBps": (dom_alg / (phases[dom] / 1e3) / 1e9) if phases[dom] > 0 else None,
                                   "note": "phases without algorithmic bytes (walk, local, sort, fold, mt ...) are the cost of making the parallel order exact"}
        roof["phase_ms_per_step"] = {k: round(v / K, 4) for k, v in phases.items()}
        roof["phase_note"] = "measured in a second identical pass with CUDA-event brackets on the engine's stream (the brackets are off in the timed pass)"

    # ---------------- cpu baseline (bounded sample, rank 0, N = 1 only) ----------------
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        threads = min(os.cpu_count() or 1, 64)
        res = run_reference(reads, args.ref_sample_reads, threads)
        if res is not None:
            cpu = {"value": res["bases"] / res["seconds"], "unit": UNIT, "cores": threads, "kind": "reference",
                   "sample": f"the first {args.ref_sample_reads} reads of the job ({res['bases'] / 1e6:.1f} Mbases), fqs-1.1 e -s -om o -qm o -im o -gs {GS} -t {threads}: 'Processing time' {res['seconds_total']:.2f} s minus {res['startup_seconds']:.2f} s of table construction (same binary on an 8-read file) = {res['seconds']:.2f} s (whole compressor, the k-mer engine is ~75% of it)"}
            if args.ref_t1_reads:
                t1 = run_reference(reads, args.ref_t1_reads, 1)
                cpu["t1_value"] = t1["bases"] / t1["seconds"]
                cpu["t1_sample"] = f"-t 1 (the parity configuration) on the first {args.ref_t1_reads} reads: {t1['seconds_total']:.2f} s minus {t1['startup_seconds']:.2f} s of table construction"

    # ---------------- whole compressor through the drop-in (bounded sample, rank 0, N = 1 only) ----------------
    compress = None
    if not args.no_compress_e2e and world == 1:
        try:
            compress = run_compress_e2e(reads, args.compress_sample_reads)
        except Exception as ex:              # never at the expense of the line itself
            compress = {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": args.warmup,
            "ms_per_step": dev_ms_max / K, "higher_is_better": True, "scaling": "strong" if sharded else "weak", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic", "config": workload_config(world, args.replicas),
            "job": {"blocks_timed": NB, "segments_timed": int(n_seg), "bases": job_bases, "device_ms": dev_ms_max, "wall_ms": wall_ms, "create_seconds": round(create_s, 3),
                    "host": {"api_ms": round((st1["api_ns"] - st0["api_ns"]) / 1e6, 1), "waiting_for_the_gpu_ms": round((st1["look_wait_ns"] - st0["look_wait_ns"]) / 1e6, 1),
                             "looks": int(st1["n_looks"] - st0["n_looks"]),
                             "note": "time of this rank inside the C-ABI calls and the part of it spent waiting for the device: the rest is launch work of the host; when the waiting share is small the early regime (thousands of ~200 us sync segments) is bound by the host's launch rate, not by the GPU"},
                    "warmup_blocks": len(warm_blocks), "warmup_note": "untimed, on a throw-away engine with its own tables: the W warm-up steps" + ("" if args.short_warmup else " and the rest of the job behind them"), "note": "table construction (fqsk_create) lies outside the timed region, as the reference's does in its arm"},
            "regimes": regimes, "roofline": roof, "parity_check": parity, "cpu_baseline": cpu, "e2e": e2e, "compress_e2e": compress, "gpu_launches": int(launches),
            "clocks": sampler.summary(), "wall_ms_per_step": wall_ms / K}
    if dumped is not None:      # the capture sits inside the timed region: this line's timings are not those of a plain run
        line["dump_outputs"] = dumped
        line["timing_comparable"] = False
        line["timing_note"] = ("--dump-outputs: every sync segment of the last step waited for a device checksum and a sampled copy of its records inside the "
                               "timed region; value, ms_per_step, regimes, job and gpu_launches are not comparable with a run without it")
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    # stdout carries the ONE JSON line and nothing else: libraries that write to file descriptor 1 (NCCL prints its version
    # there when the first communicator is created) are sent to stderr, the JSON line goes to the saved descriptor
    sys.stdout.flush()
    _real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = _real_stdout
    try:
        rc = main()
    finally:
        _real_stdout.flush()
    sys.exit(rc)
