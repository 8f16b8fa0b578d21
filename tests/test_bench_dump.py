"""CPU tests of bench.py --dump-outputs: the dumped arrays are the BWT's symbols at the dumped rows, the sample of a
large BWT is fixed and within the size limit."""
import os

import numpy as np

import bench
from oracle import coracle, stages as st
from tests.util import golden


def load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_small_bwt_has_every_row(tmp_path):
    recs = golden()["small"]["pathological"]["records"]
    sym, _ = st.text_from_records(recs)
    words, sharp, dollar = coracle.bwt(sym)
    info = bench.dump_outputs(str(tmp_path), words, sharp, dollar, sym.size)
    out = load(tmp_path)
    assert info["rows_sampled"] == sym.size
    assert out["bwt_codes"].dtype == np.float32 and out["bwt_rows"].dtype == np.float64
    assert (out["bwt_rows"] == np.arange(sym.size)).all()
    assert (out["bwt_codes"] == coracle.bwt_symbols(sym)).all()
    assert (out["sharp_rows"] == sharp.astype(np.float64)).all() and sharp.size == len(recs) - 1
    assert out["dollar_row"].dtype == np.float64 and out["dollar_row"][0] == float(dollar[0])


def test_dump_large_bwt_is_a_fixed_sample(tmp_path):
    n = bench.DUMP_ROWS * 2 + 7
    rng = np.random.default_rng(1)
    words = rng.integers(0, 2**64, size=(n + 31) // 32, dtype=np.uint64)
    sharp = np.sort(rng.choice(n, size=50, replace=False)).astype(np.uint64)
    dollar = np.array([n - 3], dtype=np.uint64)
    bench.dump_outputs(str(tmp_path / "a"), words, sharp, dollar, n)
    bench.dump_outputs(str(tmp_path / "b"), words, sharp, dollar, n)
    a, b = load(tmp_path / "a"), load(tmp_path / "b")
    assert sorted(a) == sorted(b) == ["bwt_codes", "bwt_rows", "dollar_row", "sharp_rows"]
    assert all((a[k] == b[k]).all() for k in a)
    assert sum(os.path.getsize(tmp_path / "a" / (k + ".npy")) for k in a) <= 64 << 20
    rows = a["bwt_rows"].astype(np.int64)
    assert rows.size == bench.DUMP_ROWS
    assert (np.diff(rows) > 0).all() and rows[0] >= 0 and rows[-1] < n
    full = coracle.unpack_bwt(words, n, sharp, dollar)
    assert (a["bwt_codes"] == full[rows]).all()
    assert (a["bwt_codes"] == 4).sum() == np.isin(sharp, rows).sum()
