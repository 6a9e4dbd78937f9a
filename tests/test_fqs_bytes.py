"""North-star check 3: a lossless `.fqs` produced from OUR per-base records is byte-identical to `fqs-1.1 -t 1` and decodes
with the reference decompressor.

How: oracle/_ref/fqs-1.1-replay is the reference compiled with ONE change (oracle/build_ref.py: build_replay): the count
vector, level, rough flag and cor_pos of every coded base come from a record file instead of the reference's own k-mer engine
(find_counts, rough searches, pushes, repairs and table updates are bypassed).  Its context model, range coders, id / quality /
meta streams and container code are untouched.  So `fqs-1.1-replay` fed with the engine's record stream IS the integration
INTEGRATION.md describes, and its output must equal the plain binary's byte for byte.

CPU leg: the records come from the oracle (validates the harness and the oracle).  GPU leg: from the CUDA engine via the C-ABI.
Both need the binaries in oracle/_ref/, built from the reference's sources, which the repository does not contain.  Where they are
absent, the GPU leg checks the records it would feed the replay binary against the oracle's records for the same reads."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

from fqsqueezer_b200 import engine as E
from fqsqueezer_b200 import synth
from oracle import oracle as O
from tests import helpers as H

REPLAY_BIN = os.path.join(os.path.dirname(O.REF_BIN), "fqs-1.1-replay")
needs_ref = pytest.mark.skipif(not (os.path.exists(O.REF_BIN) and os.path.exists(REPLAY_BIN)), reason="oracle/_ref binaries not built")

# (gs, genome, reads, read length, seed, N fraction, duplicate fraction)
CASES = [(1, 6000, 4000, 100, 21, 0.002, 0.01), (100, 40000, 3000, 150, 22, 0.0, 0.0)]


def _make_fastq(tmp, gs, G, n, L, seed, n_frac, dup_frac):
    genome = synth.make_genome(G, seed)
    codes, err = synth.make_reads(genome, n, L=L, seed=seed, n_frac=n_frac, dup_frac=dup_frac)
    fq = os.path.join(tmp, "in.fastq")
    synth.write_fastq(fq, codes, err, seed=seed)
    return fq


def _check(engine, gs, tmp, fq):
    base = ["e", "-s", "-om", "o", "-qm", "o", "-im", "o", "-t", "1", "-gs", str(gs), "-v", "0"]
    plain = os.path.join(tmp, "plain.fqs")
    subprocess.run([O.REF_BIN, *base, "-out", plain, fq], check=True, cwd=tmp, stdout=subprocess.DEVNULL)
    slab = np.fromfile(fq, dtype=np.uint8)
    recs = H.run_se(engine, slab)
    recs = np.ascontiguousarray(recs[recs["pos"] < 0xFFFFFFF0])
    rec_path = os.path.join(tmp, "recs.bin")
    recs.tofile(rec_path)
    ours = os.path.join(tmp, "ours.fqs")
    r = subprocess.run([REPLAY_BIN, *base, "-out", ours, fq], cwd=tmp, env=dict(os.environ, FQS_REPLAY=rec_path), capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-400:]
    a, b = open(plain, "rb").read(), open(ours, "rb").read()
    assert len(a) > 1000
    assert a == b, f".fqs differs: {len(a)} vs {len(b)} bytes, first difference at {next((i for i in range(min(len(a), len(b))) if a[i] != b[i]), -1)}"
    dec = os.path.join(tmp, "dec.fastq")
    subprocess.run([O.REF_BIN, "d", "-out", dec, ours], check=True, cwd=tmp, stdout=subprocess.DEVNULL)
    assert open(dec, "rb").read() == slab.tobytes(), "the reference decompressor does not reproduce the input"
    return len(recs), len(a)


@needs_ref
@pytest.mark.parametrize("case", CASES[:1])
def test_fqs_bytes_from_oracle_records(case):
    gs = case[0]
    pref, p, s, b = E.kmer_params(gs)
    with tempfile.TemporaryDirectory() as tmp:
        fq = _make_fastq(tmp, *case)
        o = O.OracleEngine(p, s, b, pref)
        _check(o, gs, tmp, fq)
        o.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_fqs_bytes_from_gpu_records(case):
    gs = case[0]
    pref, p, s, b = E.kmer_params(gs)
    with tempfile.TemporaryDirectory() as tmp:
        fq = _make_fastq(tmp, *case)
        e = E.KmerEngine(p, s, b, pref)
        if not (os.path.exists(O.REF_BIN) and os.path.exists(REPLAY_BIN)):
            slab = np.fromfile(fq, dtype=np.uint8)
            o = O.OracleEngine(p, s, b, pref)
            got, want = H.run_se(e, slab), H.run_se(o, slab)
            H.assert_recs_equal(got, want[want["pos"] < 0xFFFFFFF0])
            assert len(got) > 1000 and e.stats()["kernel_launches"] > 0
            e.close(); o.close()
            return
        n_recs, n_bytes = _check(e, gs, tmp, fq)
        assert e.stats()["kernel_launches"] > 0
        e.close()
