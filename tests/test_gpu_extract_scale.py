"""Extract at the size limit of one device call: the whole text inverted, and intervals across the u32 boundaries of the
index (2^31, 2^32 - 2^16) and up to N, on the C3-like text of tests/test_gpu_scale.py.  Needs the memory of that file's
whole-path cases; skips, naming the amount, when it is not free."""
import numpy as np
import pytest
import torch

from debwt_b200 import api
from tests.test_gpu_scale import _need, _text_c3_at_limit, n_max

pytestmark = [pytest.mark.gpu, pytest.mark.slow]


def test_extract_at_limit():
    _need(116, 25)
    text, seps = _text_c3_at_limit()
    n, R = text.numel(), seps.size
    assert n == n_max(R) and n > (1 << 32) - (1 << 16)
    with api.BwtBuilder(0) as b:
        b.set_text_device(text.data_ptr(), n, seps)
        b.build()
        words, sharp, dollar = b.result()
    tnp = text.cpu().numpy()
    del text
    torch.cuda.empty_cache()

    with api.BwtBuilder(0) as c:                               # a loaded result: the text is never passed in
        c.set_result(words, n, sharp, dollar)
        c.sample_sa(32)
        got = c.text()
        assert got.size == n
        bad = np.flatnonzero(got != tnp)
        assert bad.size == 0, f"text() differs from T at {bad.size} positions, first {bad[:5].tolist()}"
        del got
        assert (c.separators() == seps).all()
        edges = [(1 << 31) - 1000, (1 << 31) - 1, 1 << 31, (1 << 32) - (1 << 16) - 777, (1 << 32) - (1 << 16)]
        starts = [e - k for e in edges for k in (0, 1, 33, 4096)] + [n - 1, n - 100, (n // 32) * 32 - 5, n - 70_000, n]
        ends = [min(e + k, n) for e in edges for k in (1, 2, 31, 5000)] + [n] * 5
        offs, out = c.extract(starts, ends)
        for i, (a, e) in enumerate(zip(starts, ends)):
            assert (out[int(offs[i]):int(offs[i + 1])] == tnp[a:e]).all(), (i, a, e)
