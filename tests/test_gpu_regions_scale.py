"""Seed extension at the size limit of one device: both strands of a genome_like text, T = n_max(24) symbols (rb above
2^31), loaded with set_result and sampled at rate 32.  For 2000 seeded reads regions() equals tests/ext_ref.py over the
same call's chains().  Needs the memory of tests/test_gpu_scale.py's whole-path cases; skips, naming the amount, when it
is not free."""
import numpy as np
import pytest
import torch

from debwt_b200 import api
from tests import chain_ref as cr
from tests import ext_ref as er
from tests.test_gpu_scale import _need, n_max
from tests.test_gpu_smem_scale import both_strands_text, seeded_reads

pytestmark = [pytest.mark.gpu, pytest.mark.slow]


def test_regions_at_limit():
    _need(116, 25)
    R = 12
    n = n_max(2 * R)
    n -= (n - 2 * R) % 2
    text, seps = both_strands_text(n, R, 13)
    assert text.numel() == n and n > (1 << 32) - (1 << 17)
    with api.BwtBuilder(0) as b:
        b.set_text_device(text.data_ptr(), n, seps)
        b.build()
        words, sharp, dollar = b.result()
    tnp = text.cpu().numpy()
    del text
    torch.cuda.empty_cache()
    reads = seeded_reads(tnp, seps, 2000, 150, 21)
    with api.BwtBuilder(0) as c:
        c.set_result(words, n, sharp, dollar)
        c.sample_sa(32)
        offs, chains, cseeds = c.chains(reads)
        r_offs, regs = c.regions(reads)
    ch, cs = cr.as_tuples(chains, cseeds)
    want = er.reference(offs.tolist(), ch, cs, reads, tnp, seps)
    assert r_offs.tolist() == want[0] and er.as_tuples(regs) == want[1]
    assert (regs["rb"] > (1 << 31)).any() and (regs["strand"] == 1).any()
    assert (regs["re"] <= np.uint64(n - 2 * R)).all()
