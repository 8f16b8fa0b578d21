"""CPU model of extract (debwt_index_extract, csrc/index.cu): the inverse samples derived from the SA samples through the
sampled-row bitvector, the rate-aligned block enumeration with its start row and skip count, and the LF walks over the
oracle's BWT.  Checked against T on the golden small cases and on random multi-record texts, at rates from 1 to above N."""
import numpy as np
import pytest

from oracle import coracle, stages as st
from tests.locate_ref import suffix_array_from_bwt
from tests.util import golden

RATES = (1, 2, 4, 32, 1024)


def sample_sa(sa, rate):
    """what debwt_index_sample_sa keeps: bits[w] = (sampled rows before word w) << 32 | sampled-row mask of w, and the
    SA values of the sampled rows in row order"""
    n = sa.size
    take = (sa % rate) == 0
    padded = np.zeros(-(-n // 32) * 32, dtype=bool)
    padded[:n] = take
    masks = (padded.reshape(-1, 32).astype(np.uint64) << np.arange(32, dtype=np.uint64)).sum(axis=1).astype(np.uint64)
    counts = padded.reshape(-1, 32).sum(axis=1)
    before = np.concatenate([[0], np.cumsum(counts)[:-1]]).astype(np.uint64)
    return (before << np.uint64(32)) | masks, sa[take].astype(np.uint32)


def isa_from_sa(bits, vals, rate, n):
    """isa_from_sa_kernel: every sampled row r writes isa[vals[k] / rate] = r, k = its rank among the sampled rows"""
    isa = np.full(-(-n // rate), -1, dtype=np.int64)
    for r in range(n):
        b = int(bits[r >> 5])
        m, bit = b & 0xFFFFFFFF, 1 << (r & 31)
        if m & bit:
            k = (b >> 32) + bin(m & (bit - 1)).count("1")
            slot = int(vals[k]) // rate
            assert isa[slot] == -1, "two rows for one inverse sample"
            isa[slot] = r
    assert (isa >= 0).all(), "an inverse sample was never written"
    return isa


def host_blocks(starts, ends, rate):
    """the host loop of debwt_index_extract: block and output offsets per interval"""
    blk, off = [0], [0]
    for a, b in zip(starts, ends):
        blk.append(blk[-1] + ((b + rate - 1) // rate - a // rate if b > a else 0))
        off.append(off[-1] + b - a)
    return blk, off


def block_of(t, starts, ends, blk, rate, n):
    """what extract_kernel derives for thread t: (interval i, lo, hi, start suffix s)"""
    i = int(np.searchsorted(blk, t, side="right")) - 1           # upper_bound - 1
    a, b = starts[i], ends[i]
    q = a // rate + (t - blk[i])
    return i, max(a, q * rate), min(b, (q + 1) * rate), min((q + 1) * rate, n)


def extract(bwt, starts, ends, rate):
    """the device logic end to end; returns the output buffer (symbol codes) and the offsets"""
    n = bwt.size
    lf = np.empty(n, dtype=np.int64)
    lf[np.argsort(bwt, kind="stable")] = np.arange(n)
    dollar_row = int(np.flatnonzero(bwt == 5)[0])
    sa = suffix_array_from_bwt(bwt).astype(np.int64)
    isa = isa_from_sa(*sample_sa(sa, rate), rate, n)
    assert isa[0] == dollar_row                                    # suffix 0 is in the '$' row
    assert (sa[isa] == np.arange(isa.size) * rate).all()
    blk, off = host_blocks(starts, ends, rate)
    out = np.full(off[-1], 255, dtype=np.uint8)
    for t in range(blk[-1]):
        i, lo, hi, s = block_of(t, starts, ends, blk, rate, n)
        assert starts[i] <= lo < hi <= ends[i] and lo // rate == (hi - 1) // rate  # non-empty, inside one rate-aligned block
        assert 0 <= s - hi < rate and s - lo <= rate                # skip count, and at most `rate` symbols read
        if hi < ends[i]:
            assert s == hi                                          # only an interval's last block skips symbols
        r = dollar_row if s == n else int(isa[s // rate])
        assert sa[r] == s % n
        p = s - 1
        while True:                                                 # r is the row of suffix p + 1
            if p < hi:
                assert out[off[i] + p - starts[i]] == 255, "a position written twice"
                out[off[i] + p - starts[i]] = bwt[r]
            if p == lo:
                break
            r = int(lf[r])
            p -= 1
    assert (out != 255).all(), "a position never written"
    return out, off


def edge_intervals(n, seps, rate, rng):
    iv = [(0, 0), (n - 1, n), (n, n), (0, n), (0, 1), (n // 2, n // 2 + 1), (n // 3, n // 3)]
    for s in seps[:3].tolist():
        iv += [(max(s - 5, 0), min(s + 6, n)), (s, s + 1)]          # across a '#' and the separator alone
    if rate >= 4 and n > rate:
        q = int(rng.integers(0, n // rate))
        iv += [(q * rate + 1, q * rate + 3), (q * rate, q * rate + rate)]   # inside one block, exactly one block
    if n > rate:
        iv += [(rate - 1, rate + 1), (n - rate - 1, n)]
    for _ in range(40):
        a = int(rng.integers(0, n + 1))
        b = min(n, a + int(rng.integers(0, 3 * rate + 50)))
        iv.append((a, b))
    return iv


def check_text(sym, seps, seed):
    bwt = coracle.bwt_symbols(sym)
    n = sym.size
    rng = np.random.default_rng(seed)
    for rate in RATES:
        iv = edge_intervals(n, np.asarray(seps), rate, rng)
        starts = [a for a, _ in iv]
        ends = [b for _, b in iv]
        out, off = extract(bwt, starts, ends, rate)
        for i, (a, b) in enumerate(iv):
            assert (out[off[i]:off[i + 1]] == sym[a:b]).all(), (rate, a, b)


@pytest.mark.parametrize("name", sorted(golden()["small"]))
def test_extract_model_small_golden(name):
    recs = [r.upper().encode() for r in golden()["small"][name]["records"]]
    sym, seps = st.text_from_records(recs)
    check_text(sym, seps, 1)


def _random_texts():
    rng = np.random.default_rng(23)
    acgt = "ACGT"
    out = []
    for n_rec in (1, 3, 12):
        out.append(["".join(acgt[i] for i in rng.integers(0, 4, int(rng.integers(33, 400)))) for _ in range(n_rec)])
    out.append(["ACGTTGCA" * 9, "ACGTTGCA" * 9, "ACGTTGCA" * 5 + "A"])    # equal records
    out.append(["A" * 60, "A" * 45, "C" + "A" * 40])
    return out


@pytest.mark.parametrize("i", range(len(_random_texts())))
def test_extract_model_random_multirecord(i):
    sym, seps = st.text_from_records(_random_texts()[i])
    check_text(sym, seps, 100 + i)


def test_block_enumeration_counts():
    """the block count per interval is ceil(b / rate) - floor(a / rate), and the blocks tile [a, b) in order"""
    n = 5000
    rng = np.random.default_rng(4)
    for rate in RATES:
        iv = [(int(a), int(min(n, a + rng.integers(0, 3000)))) for a in rng.integers(0, n + 1, 200)] + [(0, n), (n, n), (7, 7)]
        starts, ends = [a for a, _ in iv], [b for _, b in iv]
        blk, _ = host_blocks(starts, ends, rate)
        covered = {}
        for t in range(blk[-1]):
            i, lo, hi, _ = block_of(t, starts, ends, blk, rate, n)
            covered.setdefault(i, []).append((lo, hi))
        for i, (a, b) in enumerate(iv):
            got = covered.get(i, [])
            assert len(got) == blk[i + 1] - blk[i]
            assert [lo for lo, _ in got[1:]] == [hi for _, hi in got[:-1]]          # contiguous, ascending
            assert (got[0][0], got[-1][1]) == (a, b) if got else a == b
