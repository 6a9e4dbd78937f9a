"""Sorted-order front end (SURVEY.md section 8 row f3): fqsk_sort_ranks against the oracle's restatement of the comparator of
CSortedFASTQFile::sort_reads (io.h:499-528), and the restatement against the REAL reference: `fqs-1.1 e -s -om s` codes the reads in the
order its own std::sort leaves them and `fqs-1.1 d` returns them in that order, so the decoded DNA lines must be the input's DNA lines
ordered by the oracle's ranks (reads of equal rank have identical DNA: the unstable sort cannot show in this comparison).
tests/golden/reference_coding_order.json keeps the SHA-256 of that decoded order, so that the comparison runs where the reference
binary is absent too (`source` says which side recorded it; FQS_RECORD_UNIT_DIGESTS=1 records it again)."""
import hashlib
import json
import os
import subprocess
import tempfile

import numpy as np
import pytest

from fqsqueezer_b200 import schedule as S
from fqsqueezer_b200 import synth
from oracle import oracle as O


def _reads(n, seed, L=60, ragged=True, n_frac=0.02, dup_frac=0.05, genome=3000):
    """A FASTQ-like slab of DNA lines: reads that overlap (shared prefixes), exact duplicates, Ns, ragged lengths down to 1 symbol."""
    rng = np.random.default_rng(seed)
    g = rng.integers(0, 4, genome).astype(np.uint8)
    lines, prev = [], None
    for _ in range(n):
        ln = int(rng.integers(1, L + 1)) if ragged and rng.random() < 0.3 else L
        st = int(rng.integers(0, max(genome // 20, 1))) * 20 % (genome - L)      # few distinct starts: long shared prefixes
        s = np.frombuffer(b"ACGT", np.uint8)[g[st:st + ln]].copy()
        s[rng.random(ln) < n_frac] = ord("N")
        if prev is not None and rng.random() < dup_frac:
            s = prev
        prev = s
        lines.append(s)
    slab = np.concatenate([np.concatenate((x, [10])).astype(np.uint8) for x in lines]) if lines else np.zeros(0, np.uint8)
    ln = np.array([len(x) for x in lines], np.uint32)
    off = np.concatenate(([0], np.cumsum(ln.astype(np.uint64) + 1)[:-1])).astype(np.uint64) if len(lines) else np.zeros(0, np.uint64)
    return slab, off, ln, lines


def _py_ranks(lines):
    nt = bytes.maketrans(bytes(range(256)), bytes(0 if c == 65 else 1 if c == 67 else 2 if c == 71 else 3 for c in range(256)))
    keys = [(bytes(x).translate(nt), bytes(x)) for x in lines]      # bytes compare: lexicographic, a proper prefix first = steps (1) + (2); then the raw bytes
    order = sorted(range(len(keys)), key=lambda i: keys[i])
    rank = np.zeros(len(keys), np.uint32)
    for pos, i in enumerate(order):
        rank[i] = rank[order[pos - 1]] if pos and keys[order[pos - 1]] == keys[i] else pos
    return rank


@pytest.mark.parametrize("n,seed", [(0, 1), (1, 2), (500, 3), (4000, 4)])
def test_oracle_ranks_follow_the_comparator(n, seed):
    slab, off, ln, lines = _reads(n, seed)
    assert np.array_equal(O.sort_ranks(slab, off, ln), _py_ranks(lines))


ORDER_DIGEST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_coding_order.json")


def test_oracle_order_is_the_order_the_reference_codes_in():
    genome = synth.make_genome(4000, 9)
    codes, err = synth.make_reads(genome, 3000, L=70, seed=9, n_frac=0.004, dup_frac=0.03)
    got = None
    with tempfile.TemporaryDirectory() as tmp:
        fq, out, dec = os.path.join(tmp, "in.fastq"), os.path.join(tmp, "x.fqs"), os.path.join(tmp, "dec.fastq")
        synth.write_fastq(fq, codes, err, seed=9)
        if os.path.exists(O.REF_BIN):
            subprocess.run([O.REF_BIN, "e", "-s", "-om", "s", "-qm", "o", "-im", "o", "-t", "1", "-gs", "1", "-v", "0", "-out", out, fq], check=True, cwd=tmp, stdout=subprocess.DEVNULL)
            subprocess.run([O.REF_BIN, "d", "-out", dec, out], check=True, cwd=tmp, stdout=subprocess.DEVNULL)
            got = open(dec, "rb").read().split(b"\n")[1::4]
        slab = np.frombuffer(open(fq, "rb").read(), np.uint8)
    off, ln, _, _ = S.parse_fastq(slab)
    rank = O.sort_ranks(slab, off, ln)
    order = np.argsort(rank, kind="stable")
    want = [bytes(slab[int(off[i]):int(off[i]) + int(ln[i])]) for i in order]
    if got is not None:
        assert got == want
    coded = got if got is not None else want
    digest = hashlib.sha256(b"\n".join(coded)).hexdigest()
    if os.environ.get("FQS_RECORD_UNIT_DIGESTS") == "1":
        src = "reference (oracle/_ref/fqs-1.1)" if got is not None else "oracle (oracle/fqs_oracle.cpp)"
        with open(ORDER_DIGEST, "w") as f:
            f.write(json.dumps({"source": src, "sha256": digest}) + "\n")
    with open(ORDER_DIGEST) as f:
        assert digest == json.load(f)["sha256"], "the order differs from the order the reference coded these reads in"


@pytest.mark.gpu
@pytest.mark.parametrize("n,seed,L", [(0, 1, 60), (1, 2, 60), (700, 3, 60), (5000, 4, 150), (120_000, 5, 100)])
def test_gpu_ranks_match_the_oracle(n, seed, L):
    from fqsqueezer_b200 import engine as E
    slab, off, ln, _ = _reads(n, seed, L=L, genome=3000 if n < 100_000 else 400_000)
    got = E.sort_ranks(slab, off, ln)
    assert np.array_equal(got, O.sort_ranks(slab, off, ln))


@pytest.mark.gpu
def test_gpu_ranks_of_one_long_run_of_equal_prefixes():
    """Thousands of reads sharing their first 32 symbols (one run of the radix key): every member is ranked against all others."""
    from fqsqueezer_b200 import engine as E
    rng = np.random.default_rng(7)
    head = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 40)]
    lines = [np.concatenate((head, np.frombuffer(b"ACGTN", np.uint8)[rng.integers(0, 5, int(rng.integers(0, 12)))])) for _ in range(3000)]
    slab = np.concatenate([np.concatenate((x, [10])).astype(np.uint8) for x in lines])
    ln = np.array([len(x) for x in lines], np.uint32)
    off = np.concatenate(([0], np.cumsum(ln.astype(np.uint64) + 1)[:-1])).astype(np.uint64)
    assert np.array_equal(E.sort_ranks(slab, off, ln), O.sort_ranks(slab, off, ln))
