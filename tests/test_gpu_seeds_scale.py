"""Seed collection at the size limit of one device: both strands of a genome_like text, T = n_max(24) symbols (rows and
positions above 2^31), loaded with set_result and sampled at rate 32.  For 2000 seeded reads round 1 equals smem(), every
seed's count equals count() of its piece, and every hit's text is its piece, with its record, strand and offset as
api.strand_offsets gives them.  Needs the memory of tests/test_gpu_scale.py's whole-path cases; skips, naming the amount,
when it is not free."""
import numpy as np
import pytest
import torch

from debwt_b200 import api
from tests.test_gpu_scale import _need, n_max
from tests.test_gpu_smem_scale import both_strands_text, seeded_reads

pytestmark = [pytest.mark.gpu, pytest.mark.slow]


def test_seeds_at_limit():
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
        offs, seeds, hits = c.seeds(reads)
        so, sm = c.smem(reads, min_len=19)
        r1 = seeds[seeds["round"] == 1]
        assert r1.size == sm.size and (r1[["row", "rc_row", "count", "qbeg", "qend"]] == sm[["row", "rc_row", "count", "qbeg", "qend"]]).all()
        owner = np.repeat(np.arange(len(reads)), np.diff(offs.astype(np.int64)))
        pieces = [reads[int(i)][int(x["qbeg"]):int(x["qend"])].upper() for i, x in zip(owner, seeds)]
        assert (c.count(pieces) == seeds["count"]).all()
        assert all((seeds["round"] == r).any() for r in (1, 2, 3))
    L = (seeds["qend"] - seeds["qbeg"]).astype(np.int64)
    lens = np.repeat(L, seeds["n_hits"].astype(np.int64))
    sid = np.repeat(np.arange(seeds.size), seeds["n_hits"].astype(np.int64))
    for h, k, s in zip(hits["pos"].tolist(), lens.tolist(), sid.tolist()):
        assert tnp[h:h + k].tobytes() == pieces[s], (s, h)
    for k in np.unique(L).tolist():
        sel = lens == k
        rec, strand, off = api.strand_offsets(hits["pos"][sel], k, seps)
        assert (rec == hits["record"][sel]).all() and (strand == hits["strand"][sel]).all() and (off == hits["offset"][sel]).all()
    assert (hits["pos"] > (1 << 31)).any()
