"""Unit-level pinning of the CPU oracle against the reference's own classes (oracle/_ref/libfqs_ref.so, a harness TU
over kmer.h / ht_kmer.h / bit_vec.h / utils.h compiled from the reference's sources by oracle/build_ref.py).

The reference side `ru` of every test is checked against tests/golden/oracle_vs_ref_units.json: the SHA-256 of every output the
reference side returned, call by call, for these seeded inputs.  Where the harness library is built, `ru` is the reference itself:
its outputs must match the stored ones and the oracle must match it.  Where it is absent (a checkout holds only the repository), `ru`
is a fresh oracle whose every output must match the stored reference output.  `source` in the file says which side recorded it:
    FQS_RECORD_UNIT_DIGESTS=1 python -m pytest tests/test_oracle_vs_ref.py
records from the reference where the harness is built, else from the oracle."""
import hashlib
import json
import os

import numpy as np
import pytest

from oracle import oracle as O

DIGESTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_vs_ref_units.json")
RECORD = os.environ.get("FQS_RECORD_UNIT_DIGESTS") == "1"
_recorded = {}


def _digest(v):
    if isinstance(v, tuple):
        return [_digest(x)[0] for x in v]
    a = np.ascontiguousarray(v)
    return [hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()[:32]]


class _Pinned:
    """The reference side of one test: every call goes to `units` and its output is compared with (or, recording, appended to) the
    stored digests of the reference's outputs, in call order.  Calls without an output (free, insert, clear) are not recorded."""

    def __init__(self, units, calls, record):
        self.units, self.calls, self.record, self.at, self.failed = units, calls, record, 0, False

    def __getattr__(self, name):
        fn = getattr(self.units, name)

        def call(*args):
            out = fn(*args)
            if out is None or name.endswith("_new"):
                return out
            d = [name, _digest(out)]
            if self.record:
                self.calls.append(d)
            else:
                self.failed = self.at >= len(self.calls) or self.calls[self.at] != d
                assert self.at < len(self.calls), f"call {self.at} ({name}): no stored reference output"
                assert self.calls[self.at] == d, f"call {self.at} ({name}): differs from the reference's stored output"
            self.at += 1
            return out
        return call


@pytest.fixture(scope="module")
def _stored():
    if RECORD:
        yield _recorded
        src = "reference (oracle/_ref/libfqs_ref.so)" if O.have_ref() else "oracle (oracle/fqs_oracle.cpp)"
        with open(DIGESTS, "w") as f:      # one line per test
            f.write('{"source": %s,\n "calls": {\n' % json.dumps(src) +
                    ",\n".join(f"  {json.dumps(k)}: {json.dumps(v)}" for k, v in sorted(_recorded.items())) + "\n}}\n")
        return
    with open(DIGESTS) as f:
        yield json.load(f)["calls"]


@pytest.fixture
def ru(request, _stored):
    units = O.ref_units() if O.have_ref() else O.oracle_units()
    if RECORD:
        _stored[request.node.name] = []
    r = _Pinned(units, _stored.get(request.node.name, []), RECORD)
    yield r
    assert RECORD or r.failed or r.at == len(r.calls), f"{r.at} reference outputs seen, {len(r.calls)} stored"


def _rand_regs(rng, k, n, cur=None):
    """n random canonical registers with `cur` symbols: returns (dir, rc, cur) left-aligned like CKmer."""
    cur = k if cur is None else cur
    syms = rng.integers(0, 4, (n, cur), dtype=np.uint64)
    d = np.zeros(n, np.uint64)
    rc = np.zeros(n, np.uint64)
    for i in range(cur):
        d |= syms[:, i] << np.uint64(62 - 2 * i)
        rc |= (np.uint64(3) - syms[:, cur - 1 - i]) << np.uint64(62 - 2 * i)
    return d, rc, np.full(n, cur, np.uint32), syms


def _normalize(d, rc, k):
    km = np.uint64(((1 << (2 * k - 8)) - 1) << (64 - 2 * k + 4))
    return np.where((d & km) < (rc & km), d, rc)


def test_mt19937_stream(ru):
    a = O.oracle_units().mt_stream(5481, 5000)
    b = ru.mt_stream(5481, 5000)
    assert np.array_equal(a, b)
    # known answers of the standard: default seed 5489 -> first output 3499211612, 10000th output 4123659995
    k = O.oracle_units().mt_stream(5489, 10000)
    assert k[0] == 3499211612 and k[9999] == 4123659995


@pytest.mark.parametrize("thr,mult,top", [(7, 2, 63), (2047, 1, 4095), (3, 1, 15)])
def test_counter_incrementer(thr, mult, top, ru):
    rng = np.random.default_rng(1)
    ou = O.oracle_units()
    co, cr = ou.cinc_new(thr, mult, top), ru.cinc_new(thr, mult, top)
    cnt = rng.integers(0, top + 1, 20000).astype(np.uint32)
    inc = rng.integers(0, top + 1, 20000).astype(np.uint32)
    assert np.array_equal(ou.cinc_inc1(co, cnt), ru.cinc_inc1(cr, cnt))
    assert np.array_equal(ou.cinc_incn(co, cnt, inc), ru.cinc_incn(cr, cnt, inc))
    small = rng.integers(0, min(top, 12) + 1, 20000).astype(np.uint32)
    assert np.array_equal(ou.cinc_incn(co, small, small[::-1].copy()), ru.cinc_incn(cr, small, small[::-1].copy()))


@pytest.mark.parametrize("k", [14, 17, 19, 24, 27])
def test_kmer_register_script(k, ru):
    rng = np.random.default_rng(k)
    ops = [(0, 0, 0)]
    cur = 0
    for _ in range(3000):
        r = rng.random()
        if cur == 0 or r < 0.45:
            ops.append((1, int(rng.integers(0, 4)), 0)); cur = min(k, cur + 1)
        elif r < 0.6:
            ops.append((2, 0, 0)); cur = min(k, cur + 1)
        elif r < 0.75:
            ops.append((3, int(rng.integers(0, 4)), 0))
        elif r < 0.9:
            ops.append((4, int(rng.integers(0, 4)), int(rng.integers(0, cur))))
        elif r < 0.95 and cur < k:
            ops.append((5, int(rng.integers(0, 4)), 0)); cur += 1
        elif r < 0.97:
            ops.append((0, 0, 0)); cur = 0
        else:
            ops.append((3, int(rng.integers(0, 4)), 0))
    ops = np.array(ops, np.uint32)
    a64, a32 = O.oracle_units().kmer_script(k, ops)
    b64, b32 = ru.kmer_script(k, ops)
    full = b32[:, 2] == 1
    # dir / rc / aligned are defined for every state; normalised / kernel only compared on full registers
    assert np.array_equal(a64[:, [0, 1, 3, 4]], b64[:, [0, 1, 3, 4]])
    assert np.array_equal(a32, b32)
    assert np.array_equal(a64[full][:, [2, 5]], b64[full][:, [2, 5]])


@pytest.mark.parametrize("k,cbits,item_bytes", [(19, 6, 4), (24, 6, 4), (27, 6, 4), (20, 12, 4), (24, 6, 8), (17, 12, 8)])
def test_table_insert_find_count(k, cbits, item_bytes, ru):
    rng = np.random.default_rng(100 + k)
    ou = O.oracle_units()
    thr, mult, top = (7, 2, 63) if cbits == 6 else (2047, 1, 4095)
    to, tr = ou.ht_new(k, cbits), ru.ht_new(k, cbits, item_bytes)
    co, cr = ou.cinc_new(thr, mult, top), ru.cinc_new(thr, mult, top)
    # a small universe so that counters climb far above thr, plus hot keys
    d, rc, cur, _ = _rand_regs(rng, k, 600)
    universe = _normalize(d, rc, k)
    stream = universe[rng.integers(0, len(universe), 40000)]
    stream = np.concatenate([stream, np.repeat(universe[:3], 3000)])
    rng.shuffle(stream)
    for part in np.array_split(stream, 5 if k < 27 else 2):      # (k = 27: the reference walks 4^13 sub-tables per dump -- two rounds are enough)
        ou.ht_insert(to, co, part)
        ru.ht_insert(tr, cr, part)
        ko, vo = ou.ht_dump(to)
        kr, vr = ru.ht_dump(tr)
        assert np.array_equal(ko, kr) and np.array_equal(vo, vr)
        # full-context lookups: registers from the universe with the placeholder in the last slot, and random misses
        qd, qrc, qcur, _ = _rand_regs(rng, k, 300)
        qd = np.concatenate([d[:300], qd]); qrc = np.concatenate([rc[:300], qrc]); qcur = np.concatenate([cur[:300], qcur])
        fo, go = ou.ht_find(to, co, k, qd, qrc, qcur)
        fr, gr = ru.ht_find(tr, cr, k, qd, qrc, qcur)
        assert np.array_equal(fo, fr) and np.array_equal(go, gr)
        assert fo.sum() > 0
        assert np.array_equal(ou.ht_count(to, universe), ru.ht_count(tr, universe))
    assert vo.max() > thr or cbits == 12
    if item_bytes == 8:      # clear(0) wipes sub-table 0 only; the 8-byte (local) tables have exactly one (ht_kmer.h:385-386, 413-417)
        ou.ht_clear(to); ru.ht_clear(tr)
        assert len(ou.ht_dump(to)[0]) == 0 and len(ru.ht_dump(tr)[0]) == 0


@pytest.mark.parametrize("k,missing", [(19, 1), (19, 2), (24, 3), (17, 4)])
def test_table_find_partial(k, missing, ru):
    """Front-truncated lookups: 4^m completions merged with PRNG-aware addition (ht_kmer.h:266-327)."""
    rng = np.random.default_rng(7 * k + missing)
    ou = O.oracle_units()
    to, tr = ou.ht_new(k, 6), ru.ht_new(k, 6, 4)
    co, cr = ou.cinc_new(7, 2, 63), ru.cinc_new(7, 2, 63)
    # universe: a few suffixes shared by many fronts so that several completions hit
    n_suf = 40
    _, _, _, suf = _rand_regs(rng, k, n_suf, cur=k - missing)
    fronts = rng.integers(0, 4, (n_suf, 6, missing), dtype=np.uint64)
    regs = []
    for i in range(n_suf):
        for f in fronts[i]:
            regs.append(np.concatenate([f, suf[i]]))
    regs = np.array(regs, np.uint64)
    d = np.zeros(len(regs), np.uint64); rc = np.zeros(len(regs), np.uint64)
    for i in range(k):
        d |= regs[:, i] << np.uint64(62 - 2 * i)
        rc |= (np.uint64(3) - regs[:, k - 1 - i]) << np.uint64(62 - 2 * i)
    keys = _normalize(d, rc, k)
    stream = keys[rng.integers(0, len(keys), 6000)]
    ou.ht_insert(to, co, stream); ru.ht_insert(tr, cr, stream)
    # queries: the truncated registers (k - missing symbols, last one is the placeholder position)
    cur = k - missing
    qd = np.zeros(n_suf, np.uint64); qrc = np.zeros(n_suf, np.uint64)
    for i in range(cur):
        qd |= suf[:, i] << np.uint64(62 - 2 * i)
        qrc |= (np.uint64(3) - suf[:, cur - 1 - i]) << np.uint64(62 - 2 * i)
    qcur = np.full(n_suf, cur, np.uint32)
    fo, go = ou.ht_find(to, co, k, qd, qrc, qcur)
    fr, gr = ru.ht_find(tr, cr, k, qd, qrc, qcur)
    assert np.array_equal(fo, fr) and np.array_equal(go, gr)
    assert fo.max() > 7      # merged counts above thr -> the PRNG path ran
    # the PRNG streams must be in the same state afterwards
    probe = np.full(64, 30, np.uint32)
    assert np.array_equal(ou.cinc_inc1(co, probe), ru.cinc_inc1(cr, probe))


def test_small_int_vector(ru):
    rng = np.random.default_rng(5)
    ou = O.oracle_units()
    bits = 24
    so, sr = ou.siv_new(bits), ru.siv_new(bits)
    idx = rng.integers(0, 1 << bits, 300000).astype(np.uint64)
    idx = np.concatenate([idx, np.repeat(idx[:100], 5)])
    assert ou.siv_increment(so, idx) == ru.siv_increment(sr, idx)
    q = rng.integers(0, 1 << bits, 5000).astype(np.uint64)
    q = np.concatenate([q, idx[:5000]])
    assert np.array_equal(ou.siv_test(so, q), ru.siv_test(sr, q))
    assert np.array_equal(ou.siv_counts(so, q), ru.siv_counts(sr, q))
    for size in (24, 22, 18, 14, 10, 8):
        pre = (q >> np.uint64(bits - size)).astype(np.uint64)
        assert np.array_equal(ou.siv_test_shorter(so, pre, np.full(len(pre), size, np.uint32)),
                              ru.siv_test_shorter(sr, pre, np.full(len(pre), size, np.uint32)))


def test_pair_table(ru):
    rng = np.random.default_rng(9)
    ou = O.oracle_units()
    k = 24
    po, pr = ou.pair_new(k), ru.pair_new(k, 1)
    vm = (1 << (2 * k)) - 1
    keys = rng.integers(0, vm, 500).astype(np.uint64)
    vals = rng.integers(0, vm, 800).astype(np.uint64)
    kk = keys[rng.integers(0, 500, 200000)]
    vv = vals[rng.integers(0, 800, 200000)]
    kk[::97] = vm          # sentinel: never inserted (ht_kmer.cpp:123-124)
    vv[::89] = vm
    cc = rng.integers(1, 5, 200000).astype(np.uint64)
    cc[::1000] = 70000     # saturates the 16-bit counter
    ou.pair_insert(po, kk, vv, cc); ru.pair_insert(pr, kk, vv, cc)
    for key in keys[:50]:
        assert np.array_equal(ou.pair_find(po, key), ru.pair_find(pr, key))
    assert np.array_equal(ou.pair_count(po, kk[:5000], vv[:5000]), ru.pair_count(pr, kk[:5000], vv[:5000]))
