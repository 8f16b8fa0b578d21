"""The sharded build (csrc/shard.cu) at its slice, splitter and row boundaries (inputs and placements in
tests/shard_points.py), at every world size from 1 to 16, with every rank's counts compared with the per-rank restatement.

The G ranks run as threads of this process, each with its own debwt_shard on cuda:0 (what debwt_build_multi does), so that
every rank's stats can be read, not just rank 0's.  A wrong owner rule at a splitter or a wrong sampling stride still
partitions the keys and leaves the BWT right: only the ranks' key counts see them, so they are compared on every rank."""
import functools
import itertools
import os
import threading

import numpy as np
import pytest

from debwt_b200 import api, binding
from tests import shard_points as sp

pytestmark = pytest.mark.gpu

_tags = itertools.count()


@pytest.fixture
def shard_threads():
    """run(G, jobs): G ranks as threads, each with its own Shard on cuda:0, build the (text, seps) jobs in order on the
    same shards.  Returns per rank and job ("ok", result, stats) or ("error", message).  Every thread is joined."""
    threads = []

    def run(G, jobs):
        tag = f"sp_{os.getpid()}_{next(_tags)}"
        out = [[None] * len(jobs) for _ in range(G)]
        fail = [None] * G

        def work(r):
            try:
                with api.Shard(0, r, G, tag, same_process=True) as sh:
                    for j, (text, seps) in enumerate(jobs):
                        try:
                            sh.build_host(text, seps)
                        except binding.DebwtError as e:
                            out[r][j] = ("error", str(e))
                            continue
                        out[r][j] = ("ok", sh.result(), sh.stats())
            except BaseException as e:  # noqa: BLE001  (reported by the test)
                fail[r] = repr(e)

        th = [threading.Thread(target=work, args=(r,), daemon=True) for r in range(G)]
        threads.extend(th)
        for t in th:
            t.start()
        for t in th:
            t.join(timeout=900)
        assert not any(t.is_alive() for t in th), "a rank did not finish"
        assert fail == [None] * G, fail
        return out

    yield run
    for t in threads:            # a rank stuck in the communicator leaves its barrier on its own after a timeout
        t.join()


@functools.lru_cache(maxsize=None)
def _restated(name):
    c = sp.CASES[name]
    return sp.Restated(c.make(), doubling=c.doubling)


@functools.lru_cache(maxsize=None)
def _single_gpu(name):
    """(words, sharp, dollar), stats of the single-GPU build"""
    text, seps = api.join_records(_restated(name).records)
    with api.BwtBuilder() as b:
        b.set_text(text, seps)
        b.build()
        return b.result(), b.stats()


def _same(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a, b))


def _check(name, G, outs):
    """one job's outcome on every rank against the restatement and the single-GPU build"""
    rs = _restated(name)
    rk = rs.ranks(G)
    assert all(o[0] == "ok" for o in outs), [o[1] for o in outs if o[0] != "ok"]
    assert _same(outs[0][1], rs.ref()), f"{name} at world {G}: BWT differs"
    want = rs.stats()
    one, one_stats = _single_gpu(name)
    assert _same(one, rs.ref())
    for r, (_, _, s) in enumerate(outs):
        assert s["n_keys_local"] == rk.n_keys_local[r], (name, G, r, [o[2]["n_keys_local"] for o in outs], rk.n_keys_local)
        assert s["sort_sweeps"] == rk.sort_sweeps[r], (name, G, r)
        for k in ("n_branch", "n_blue", "n_codes"):
            assert s[k] == want[k] == one_stats[k], (name, G, r, k)
        assert s["n_keys"] == want["n_keys"] and s["n_symbols"] == rs.n and s["n_records"] == rs.R


def _params():
    return [pytest.param(n, G, id=f"{n}-g{G}") for n, c in sp.CASES.items() for G in c.worlds]


@pytest.mark.parametrize("name,G", _params())
def test_shard_point(name, G, shard_threads):
    case = sp.CASES[name]
    rs = _restated(name)
    case.place(rs)
    text, seps = api.join_records(rs.records)
    # a second input on the same shards: smaller after a large case, larger after a small one
    other = "in_edges" if rs.n > _restated("in_edges").n else "grid_7_8"
    o_text, o_seps = api.join_records(_restated(other).records)
    outs = shard_threads(G, [(text, seps), (o_text, o_seps)])
    _check(name, G, [o[0] for o in outs])
    o_outs = [o[1] for o in outs]
    assert all(o[0] == "ok" for o in o_outs) and _same(o_outs[0][1], _restated(other).ref()), f"{other} after {name} at world {G}"
    assert [o[2]["n_keys_local"] for o in o_outs] == _restated(other).ranks(G).n_keys_local
    # debwt_build_multi: the same bytes, rank 0's stats
    w, s, d, stats = api.build_multi(text, seps, [0] * G)
    assert _same((w, s, d), outs[0][0][1])
    assert stats["n_keys_local"] == outs[0][0][2]["n_keys_local"] and stats["n_codes"] == outs[0][0][2]["n_codes"]


def _bad_inputs(rs, rk):
    text, seps = api.join_records(rs.records)
    G = rk.G
    bad_base = text.copy()
    p = rk.pos_lo[G - 1] + 10
    assert chr(bad_base[p]) in "ACGT"
    bad_base[p] = ord("N")                                           # in the last rank's slice only
    bad_sep = text.copy()
    p = rk.pos_lo[2] + 100
    assert chr(bad_sep[p]) in "ACGT" and rk.pos_hi[2] > p
    bad_sep[p] = ord("#")                                            # inside a record, in a middle rank's slice only
    short = api.join_records(rs.records[:-1] + [rs.records[-1][:32]])
    last = seps.copy()
    last[-1] -= 1
    return [((bad_base, seps), "symbol other than A, C, G, T"), ((bad_sep, seps), "reserved for the record separators"),
            (short, "Length <= 32"), ((text, last), "last separator must be the last symbol")]


def test_errors_on_every_rank_then_a_valid_build(shard_threads):
    name, G = "sep_edges_g5", 5
    rs = _restated(name)
    rk = rs.ranks(G)
    good = api.join_records(rs.records)
    bad = _bad_inputs(rs, rk)
    jobs = [j for inp, _ in bad for j in (inp, good)]
    outs = shard_threads(G, jobs)
    for b, (_, msg) in enumerate(bad):
        errs = [outs[r][2 * b] for r in range(G)]
        assert all(e[0] == "error" for e in errs), (msg, errs)
        assert len({e[1] for e in errs}) == 1 and msg in errs[0][1], (msg, errs)
        _check(name, G, [outs[r][2 * b + 1] for r in range(G)])


def test_world_17_is_refused():
    with pytest.raises(binding.DebwtError, match="1..16 ranks"):
        api.Shard(0, 0, 17, f"sp17_{os.getpid()}", same_process=True)
    text, seps = api.join_records(_restated("sep_edges_g5").records)
    with pytest.raises(binding.DebwtError, match="bad argument"):
        api.build_multi(text, seps, [0] * 17)
