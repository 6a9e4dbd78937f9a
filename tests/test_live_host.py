"""The drop-in, compiled: host/_bin/fqs-1.1-fqsk is the reference compressor with its k-mer engine replaced by the C-ABI of
include/fqsk.h (host/build_host.py + host/fqsk_live.h; INTEGRATION.md).  It binds the library with dlopen($FQSK_LIB).

CPU leg : $FQSK_LIB = a mock built from the oracle (tests/mock_fqsk.cpp).  Checks the HOST half -- the patched worker loop
          (segment boundaries, block starts, end-of-block syncs) and compress_suffix consuming records.
GPU leg : $FQSK_LIB = fqsqueezer_b200/libfqsk.so.  The whole thing: reads_block slabs -> fqsk_segment / fqsk_sync on the B200 ->
          the reference's context model and range coders.
Both: the .fqs is byte-identical to the unmodified `fqs-1.1 -t 1` and the unmodified binary decodes it back to the input.
The binaries (host/_bin, oracle/_ref) are built from the reference's sources, which the repository does not contain.  Where they are
absent, the GPU legs check the engine half of the same run instead (_engine_half)."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

from fqsqueezer_b200 import engine as E
from fqsqueezer_b200 import schedule as S
from fqsqueezer_b200 import synth
from oracle import oracle as O
from tests import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIVE_BIN = os.path.join(ROOT, "host", "_bin", "fqs-1.1-fqsk")
REAL_LIB = os.path.join(ROOT, "fqsqueezer_b200", "libfqsk.so")
HAVE_BINS = os.path.exists(O.REF_BIN) and os.path.exists(LIVE_BIN)
needs_bins = pytest.mark.skipif(not HAVE_BINS, reason="host/_bin or oracle/_ref not built")


def _fastq_records(path):
    slab = np.fromfile(path, np.uint8)
    _, _, roff, rsz = S.parse_fastq(slab)
    return [slab[int(a):int(a) + int(n)] for a, n in zip(roff, rsz)]


def _engine_half(files, gs, layout=("-s", "-om", "o"), submit=False):
    """The engine half of a drop-in run, for a checkout without the binaries: the reads of `files` in the order the drop-in hands them to
    libfqsk.so (pairs interleaved; in sorted order (-om s) ordered by the comparator of CSortedFASTQFile::sort_reads, of mate 1 when
    paired), through the C-ABI on the GPU -- fqsk_submit / fqsk_collect when `submit`, else fqsk_segment / fqsk_sync -- against the CPU
    oracle on the same schedule (pinned to the tapped reference by test_golden_oracle): records, pair decisions, sorted-prefix flags and
    difs and every table, bit-exact."""
    paired, srt = layout[0] == "-p", layout[-1] == "s"
    recs = [_fastq_records(f) for f in files]
    recs = [r for pair in zip(*recs) for r in pair] if paired else recs[0]
    step = 2 if paired else 1
    if srt:
        first = np.concatenate(recs[0::step])
        off, ln, _, _ = S.parse_fastq(first)
        order = np.argsort(O.sort_ranks(first, off, ln), kind="stable")
        recs = [r for i in order for r in recs[step * i:step * i + step]]
    slab = np.concatenate(recs)
    mode = (2 if paired else 0) + (1 if srt else 0)
    pref, p, s, b = E.kmer_params(gs)
    e = E.KmerEngine(p, s, b, pref, mode=mode)
    o = O.OracleEngine(p, s, b, pref, mode=mode)
    if submit:
        assert not srt
        got = H.run_async(e, slab, paired=paired)
        got = (got[0], got[2]) if paired else got[:1]
        want = H.run_pe(o, slab) if paired else (H.run_se(o, slab),)
    else:
        run = {0: lambda x, g: (H.run_se(x, slab),), 1: lambda x, g: H.run_sorted(x, slab, g), 2: lambda x, g: H.run_pe(x, slab, g),
               3: lambda x, g: H.run_pe_sorted(x, slab, g)}[mode]
        got, want = run(e, True), run(o, False)
    H.assert_recs_equal(got[0], want[0][want[0]["pos"] < 0xFFFFFFF0])
    assert len(got[0]) > 1000
    for i in range(1, len(want)):
        assert np.array_equal(got[i], want[i]), i
    for which in range(4 if paired else 3):
        kg, vg = e.dump(which)
        ko, vo = o.dump(which)
        assert np.array_equal(kg, ko) and np.array_equal(vg, vo), which
    assert e.stats()["kernel_launches"] > 0
    e.close(); o.close()


# (gs, genome, reads, read length, seed, N fraction, duplicate fraction)
CASES = [(1, 6000, 4000, 100, 31, 0.002, 0.01), (100, 40000, 3000, 150, 32, 0.0, 0.0)]
# > 1 reads_block (16 MiB slabs): block starts, decreasing sync counts, end-of-block syncs
BIG = (100, 400000, 60000, 150, 33, 0.0005, 0.002)


def _fastq(tmp, gs, G, n, L, seed, n_frac, dup_frac):
    genome = synth.make_genome(G, seed)
    codes, err = synth.make_reads(genome, n, L=L, seed=seed, n_frac=n_frac, dup_frac=dup_frac)
    fq = os.path.join(tmp, "in.fastq")
    synth.write_fastq(fq, codes, err, seed=seed)
    return fq


def _fastq_pe(tmp, gs, G, n_pairs, L, seed):
    genome = synth.make_genome(G, seed)
    c1, e1, c2, e2 = synth.make_pairs(genome, n_pairs, L=L, seed=seed, ins_mean=2.2 * L, ins_sd=0.2 * L)
    f1, f2 = os.path.join(tmp, "in_1.fastq"), os.path.join(tmp, "in_2.fastq")
    synth.write_fastq(f1, c1, e1, mate=1, seed=seed)
    synth.write_fastq(f2, c2, e2, mate=2, seed=seed + 1)
    return f1, f2


def _build_mock(tmp):
    O.build_oracle()
    so = os.path.join(tmp, "libfqsk_mock.so")
    odir = os.path.dirname(O.ORACLE_SO)
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", os.path.join(ROOT, "tests", "mock_fqsk.cpp"), "-I", os.path.join(ROOT, "include"),
                    "-L", odir, "-l:libfqs_oracle.so", f"-Wl,-rpath,{odir}", "-o", so], check=True)
    return so


def _check(lib, gs, tmp, fq, decode=True, layout=("-s", "-om", "o"), threads=1, env=None):
    """fq: one FASTQ path (single-end) or a pair of paths (paired-end).  layout: the reference's read layout / order options.
    threads: the reference's -t (the live host runs one engine per worker thread; the comparison is with `fqs-1.1 -t threads`)."""
    files = [fq] if isinstance(fq, str) else list(fq)
    base = ["e", *layout, "-qm", "o", "-im", "o", "-t", str(threads), "-gs", str(gs), "-v", "0"]
    plain, ours = os.path.join(tmp, "plain.fqs"), os.path.join(tmp, "ours.fqs")
    subprocess.run([O.REF_BIN, *base, "-out", plain, *files], check=True, cwd=tmp, stdout=subprocess.DEVNULL)
    r = subprocess.run([LIVE_BIN, *base, "-out", ours, *files], cwd=tmp, env=dict(os.environ, FQSK_LIB=lib, FQSK_VERBOSE="1", **(env or {})), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-600:]
    a, b = open(plain, "rb").read(), open(ours, "rb").read()
    assert len(a) > 1000
    assert a == b, f".fqs differs: {len(a)} vs {len(b)} bytes, first difference at {next((i for i in range(min(len(a), len(b))) if a[i] != b[i]), -1)}"
    if decode and len(files) == 1:
        dec = os.path.join(tmp, "dec.fastq")
        subprocess.run([O.REF_BIN, "d", "-out", dec, ours], check=True, cwd=tmp, stdout=subprocess.DEVNULL)
        got, want = open(dec, "rb").read(), open(fq, "rb").read()
        if "s" == layout[-1]:      # sorted order: the decoder returns the reads in the order they were coded
            assert sorted(got.split(b"\n")[1::4]) == sorted(want.split(b"\n")[1::4]), "the reference decompressor lost reads"
        else:
            assert got == want, "the reference decompressor does not reproduce the input"
    return r.stderr


# other modes of the live host: sorted order (-om s: compress_prefix_sorted's flag / dif from the engine) and paired end (-p:
# CompressPE's shared-minimizer decision from the engine); (gs, genome, reads or pairs, read length, seed)
SORTED = [(1, 5000, 2500, 70, 45), (16, 60000, 6000, 150, 46)]
PAIRED = [(1, 5000, 1200, 80, 71), (100, 50000, 4000, 150, 72)]
# -p in the reference's DEFAULT order (-om s, params.h:60): BASELINE configs 3 and 5 as literally written
PAIRED_SORTED = [(1, 5000, 1500, 80, 73), (100, 50000, 4000, 150, 74)]


def _engine_half_of(case, layout):
    """_engine_half on the input _run_sorted / _run_paired generate for `case`."""
    gs, G, n, L, seed = case
    with tempfile.TemporaryDirectory() as tmp:
        files = _fastq_pe(tmp, gs, G, n, L, seed) if layout[0] == "-p" else [_fastq(tmp, gs, G, n, L, seed, 0.002, 0.01)]
        _engine_half(files, gs, layout)


def _run_sorted(lib, case):
    gs, G, n, L, seed = case
    with tempfile.TemporaryDirectory() as tmp:
        fq = _fastq(tmp, gs, G, n, L, seed, 0.002, 0.01)
        return _check(lib(tmp), gs, tmp, fq, layout=("-s", "-om", "s"))


def _run_paired(lib, case, order="o"):
    gs, G, n, L, seed = case
    with tempfile.TemporaryDirectory() as tmp:
        return _check(lib(tmp), gs, tmp, _fastq_pe(tmp, gs, G, n, L, seed), layout=("-p", "-om", order))


@needs_bins
@pytest.mark.parametrize("case", SORTED)
def test_live_host_sorted_with_oracle_records(case):
    assert "segments" in _run_sorted(_build_mock, case)


@needs_bins
@pytest.mark.parametrize("case", PAIRED)
def test_live_host_paired_with_oracle_records(case):
    assert "segments" in _run_paired(_build_mock, case)


# (CPU leg at -gs 16: compress_prefix_sorted's linear scan between consecutive p-mers -- in the reference AND in the oracle -- covers 4^p fields
#  per bin pass; p = 17 costs two minutes of host time for nothing the p = 15 run does not exercise.  The GPU leg keeps -gs 100.)
@needs_bins
@pytest.mark.parametrize("case", [PAIRED_SORTED[0], (16, 50000, 4000, 150, 74)])
def test_live_host_paired_sorted_with_oracle_records(case):
    assert "segments" in _run_paired(_build_mock, case, order="s")


@pytest.mark.gpu
@pytest.mark.parametrize("case", PAIRED_SORTED)
def test_live_host_paired_sorted_on_gpu(case):
    if not HAVE_BINS:
        return _engine_half_of(case, ("-p", "-om", "s"))
    log = _run_paired(lambda tmp: REAL_LIB, case, order="s")
    assert "kernel launches" in log and " 0 kernel launches" not in log, log


@needs_bins
def test_live_host_paired_multi_block_with_oracle_records():
    """Paired end over more than one reads_block (two 16 MiB slabs per block, application.cpp:1057-1104): block starts, the
    i >= next_synchro rule with i stepping by 2, end-of-block syncs."""
    assert "segments" in _run_paired(_build_mock, (100, 400000, 35000, 150, 91))


@pytest.mark.gpu
@pytest.mark.parametrize("case", SORTED)
def test_live_host_sorted_on_gpu(case):
    if not HAVE_BINS:
        return _engine_half_of(case, ("-s", "-om", "s"))
    log = _run_sorted(lambda tmp: REAL_LIB, case)
    assert "kernel launches" in log and " 0 kernel launches" not in log, log


@pytest.mark.gpu
@pytest.mark.parametrize("case", PAIRED)
def test_live_host_paired_on_gpu(case):
    if not HAVE_BINS:
        return _engine_half_of(case, ("-p", "-om", "o"))
    log = _run_paired(lambda tmp: REAL_LIB, case)
    assert "kernel launches" in log and " 0 kernel launches" not in log, log


@needs_bins
@pytest.mark.parametrize("case", CASES + [BIG])
def test_live_host_with_oracle_records(case):
    with tempfile.TemporaryDirectory() as tmp:
        fq = _fastq(tmp, *case)
        log = _check(_build_mock(tmp), case[0], tmp, fq, decode=case is not BIG)
        assert "segments" in log


def _make_ragged(fq, seed, lo):
    """Cuts half of the reads to a random length in [lo, L] (DNA and quality lines alike)."""
    rng = np.random.default_rng(seed)
    lines = open(fq, "rb").read().split(b"\n")
    out = []
    for i in range(0, len(lines) - 1, 4):
        L = len(lines[i + 1])
        k = int(rng.integers(lo, L + 1)) if rng.random() < 0.5 else L
        out += [lines[i], lines[i + 1][:k], lines[i + 2], lines[i + 3][:k]]
    open(fq, "wb").write(b"\n".join(out) + b"\n")


@needs_bins
@pytest.mark.parametrize("lo", [25, 3])
def test_live_host_ragged_reads_with_oracle_records(lo):
    """Reads of unequal length, down to reads shorter than the directly coded prefix (prefix_len = 9 at -gs 1): descriptors,
    record capacity and the record cursor of the binding must follow the reference's own walk over such reads."""
    with tempfile.TemporaryDirectory() as tmp:
        fq = _fastq(tmp, 1, 6000, 3000, 100, 77, 0.003, 0.01)
        _make_ragged(fq, 5, lo)
        assert "segments" in _check(_build_mock(tmp), 1, tmp, fq)


@pytest.mark.gpu
@pytest.mark.parametrize("lo", [25, 3])
def test_live_host_ragged_reads_on_gpu(lo):
    with tempfile.TemporaryDirectory() as tmp:
        fq = _fastq(tmp, 1, 6000, 3000, 100, 77, 0.003, 0.01)
        _make_ragged(fq, 5, lo)
        if not HAVE_BINS:
            return _engine_half([fq], 1)
        log = _check(REAL_LIB, 1, tmp, fq)
        assert "kernel launches" in log and " 0 kernel launches" not in log, log


def _run_golden_fqs(lib, name, tmp):
    """The compiled drop-in on the FASTQ of a golden fixture; its .fqs must equal the reference's own, which rides in the fixture
    (at -gs 3100 the reference needs 45 GB and a minute of table construction per run: it ran once, in oracle/make_golden.py)."""
    from tests import helpers as H
    g = H.load_golden(name)
    extra = [str(x) for x in g["extra"]]
    fq = os.path.join(tmp, "in.fastq")
    lines = g["fastq"].tobytes().split(b"\n")
    if "-p" in extra:      # the fixture holds the pairs interleaved
        recs = [lines[i:i + 4] for i in range(0, len(lines) - 1, 4)]
        f1, f2 = os.path.join(tmp, "in_1.fastq"), os.path.join(tmp, "in_2.fastq")
        open(f1, "wb").write(b"".join(b"\n".join(r) + b"\n" for r in recs[0::2]))
        open(f2, "wb").write(b"".join(b"\n".join(r) + b"\n" for r in recs[1::2]))
        files, layout = [f1, f2], extra
    else:
        open(fq, "wb").write(g["fastq"].tobytes())
        files, layout = [fq], ["-s", *extra]
    ours = os.path.join(tmp, "ours.fqs")
    base = ["e", *layout, "-qm", "o", "-im", "o", "-t", "1", "-gs", str(int(g["gs"])), "-v", "0"]
    r = subprocess.run([LIVE_BIN, *base, "-out", ours, *files], cwd=tmp, env=dict(os.environ, FQSK_LIB=lib, FQSK_VERBOSE="1"), capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-600:]
    a, b = g["fqs"].tobytes(), open(ours, "rb").read()
    assert len(a) > 1000
    assert a == b, f".fqs differs: {len(a)} vs {len(b)} bytes, first difference at {next((i for i in range(min(len(a), len(b))) if a[i] != b[i]), -1)}"
    return r.stderr


@pytest.mark.skipif(not os.path.exists(LIVE_BIN), reason="host/_bin not built")
@pytest.mark.parametrize("name", ["se_orig_gs3100", "pe_orig_gs3100"])
def test_live_host_default_kmer_lengths_with_oracle_records(name):
    """-gs 3100 (the reference's default: p18/s21/b27, prefix 13) through the compiled drop-in, oracle behind the ABI."""
    with tempfile.TemporaryDirectory() as tmp:
        assert "segments" in _run_golden_fqs(_build_mock(tmp), name, tmp)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["se_orig_gs3100", "pe_orig_gs3100"])
def test_live_host_default_kmer_lengths_on_gpu(name):
    if not os.path.exists(LIVE_BIN):      # the engine half against the reference's own records, which ride in the fixture
        g = H.load_golden(name)
        pref, p, s, b = E.kmer_params(int(g["gs"]))
        paired = "-p" in [str(x) for x in g["extra"]]
        e = E.KmerEngine(p, s, b, pref, mode=E.MODE_PE_ORIGINAL if paired else E.MODE_SE_ORIGINAL)
        if paired:
            recs, info = H.run_pe(e, g["fastq"], is_gpu=True)
            want, winfo = H.golden_pe_expect(g)
            assert np.array_equal(info, winfo)
        else:
            recs, want = H.run_se(e, g["fastq"]), g["recs"][g["recs"]["pos"] < 0xFFFFFFF0]
        H.assert_recs_equal(recs, want)
        H.assert_dump_equal(e, g, pairs=paired)
        e.close()
        return
    with tempfile.TemporaryDirectory() as tmp:
        log = _run_golden_fqs(REAL_LIB, name, tmp)
        assert "kernel launches" in log and " 0 kernel launches" not in log, log


@needs_bins
def test_live_host_fails_loudly_without_engine():
    """No CPU fallback: without a loadable library the compressor stops before it writes anything."""
    with tempfile.TemporaryDirectory() as tmp:
        fq = _fastq(tmp, *CASES[0])
        r = subprocess.run([LIVE_BIN, "e", "-s", "-om", "o", "-t", "1", "-gs", "1", "-v", "0", "-out", os.path.join(tmp, "x.fqs"), fq], cwd=tmp,
                           env=dict(os.environ, FQSK_LIB=os.path.join(tmp, "missing.so")), capture_output=True, text=True)
        assert r.returncode == 3 and "no CPU fallback" in r.stderr.replace("There is no", "no")
        # modes the live host does not cover (more worker threads than the 8 GPUs of a box) stop the same way (never silently served by the CPU classes)
        r = subprocess.run([LIVE_BIN, "e", "-s", "-om", "o", "-t", "9", "-gs", "1", "-v", "0", "-out", os.path.join(tmp, "x.fqs"), fq], cwd=tmp,
                           env=dict(os.environ, FQSK_LIB=_build_mock(tmp)), capture_output=True, text=True)
        assert r.returncode == 3 and "no CPU fallback" in r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("layout,case", [(("-s", "-om", "o"), CASES[0]), (("-p", "-om", "o"), PAIRED[0])])
def test_live_host_count_records_on_gpu(layout, case, monkeypatch):
    """The GPU legs of this file run with the 16-byte context records built on the device (fqsk_submit_ctx, the binding's default when
    the library exports it: the log says so); this one keeps the 28-byte count-record path (FQSK_CTX=0, host-side determine_ctx_codes)
    covered on the GPU as well.  Both must give the reference's bytes."""
    monkeypatch.setenv("FQSK_CTX", "0")
    with tempfile.TemporaryDirectory() as tmp:
        if not HAVE_BINS:      # the 28-byte count records through fqsk_submit / fqsk_collect
            gs, G, n, L, seed = case[:5]
            files = _fastq_pe(tmp, gs, G, n, L, seed) if layout[0] == "-p" else [_fastq(tmp, *case)]
            return _engine_half(files, gs, layout, submit=True)
        if layout[0] == "-p":
            gs, G, n, L, seed = case
            log = _check(REAL_LIB, gs, tmp, _fastq_pe(tmp, gs, G, n, L, seed), layout=layout)
        else:
            log = _check(REAL_LIB, case[0], tmp, _fastq(tmp, *case), layout=layout)
        assert "28-byte count records" in log, log


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES + [BIG])
def test_live_host_on_gpu(case):
    assert os.path.exists(REAL_LIB), "fqsqueezer_b200/libfqsk.so is not built"
    with tempfile.TemporaryDirectory() as tmp:
        fq = _fastq(tmp, *case)
        if not HAVE_BINS:      # over several reads_blocks too (BIG), through fqsk_submit / fqsk_collect
            return _engine_half([fq], case[0], submit=True)
        log = _check(REAL_LIB, case[0], tmp, fq, decode=case is not BIG)
        assert "kernel launches" in log and " 0 kernel launches" not in log, log
        assert "16-byte context records built on the device" in log, log


# ---- -t N: one engine per worker thread (host/fqsk_live.h), tables hash-sharded over the engines; the .fqs must equal `fqs-1.1 -t N` ----
# (layout, gs, genome, reads or pairs, read length, seed, threads)
WORKERS = [(("-s", "-om", "o"), 1, 6000, 4000, 100, 131, 2), (("-s", "-om", "s"), 1, 5000, 2500, 70, 145, 2), (("-p", "-om", "o"), 1, 5000, 1200, 80, 171, 2),
           (("-p", "-om", "s"), 1, 5000, 1500, 80, 173, 2), (("-s", "-om", "o"), 16, 30000, 5000, 120, 132, 3)]


def _run_workers(lib, case, env=None):
    layout, gs, G, n, L, seed, T = case
    with tempfile.TemporaryDirectory() as tmp:
        fq = _fastq_pe(tmp, gs, G, n, L, seed) if layout[0] == "-p" else _fastq(tmp, gs, G, n, L, seed, 0.002, 0.01)
        return _check(lib(tmp), gs, tmp, fq, layout=layout, threads=T, env=env)


@needs_bins
@pytest.mark.parametrize("case", WORKERS)
def test_live_host_worker_threads_with_oracle_records(case):
    """The worker loop at -t N over the C-ABI (application.cpp:575-671 / 1105-1193): every worker thread binds its own engine, codes its slice of
    every reads_block from that engine's records and meets the others in the sync.  CPU leg: the mock serves N oracle workers on shared
    tables (the reference's -t N semantics)."""
    log = _run_workers(_build_mock, case)
    assert log.count("segments") == case[-1], log


@needs_bins
def test_live_host_worker_threads_multi_block_with_oracle_records():
    """-t 2 over several reads_blocks: PartitionForWorkers per block (reads_block.h:197-214), the sync count of a block falling with its
    generation and with the worker's share (application.h:85-92), end-of-block syncs of both workers."""
    log = _run_workers(_build_mock, (("-s", "-om", "o"), 100, 400000, 60000, 150, 133, 2))
    assert log.count("segments") == 2, log


def _n_gpus():
    try:      # (no torch import: this file drives compiled binaries only)
        return len([x for x in subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True, timeout=30).stdout.splitlines() if x.startswith("GPU ")])
    except Exception:
        return 0


@needs_bins
@pytest.mark.gpu
@pytest.mark.parametrize("case", WORKERS[:4])
@pytest.mark.parametrize("grow", [False, True])
def test_live_host_worker_threads_on_gpus(case, grow):
    """-t 2 on two B200s: one sharded engine per worker thread in ONE process (fqsk_shard_attach_local: peer access instead of IPC),
    fqsk_segment + fqsk_sync_device per sync segment; .fqs byte-identical to `fqs-1.1 -t 2`.  grow: smallest tables, crowded at 1/64 of the
    usual load -- the shards double together several times (FQSK_RESHARD handled by the worker threads)."""
    if _n_gpus() < case[-1]:
        pytest.skip(f"needs {case[-1]} GPUs")
    env = dict(FQSK_LOG2_BUCKETS="1", FQSK_PAIR_LOG2_SLOTS="10", FQSK_FLAGS=str(4 | 32)) if grow else None
    log = _run_workers(lambda tmp: REAL_LIB, case, env=env)
    assert "kernel launches" in log and " 0 kernel launches" not in log, log
    if grow:
        assert " 0 coordinated table doublings" not in log, log
