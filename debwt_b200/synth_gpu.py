"""The synthetic genomes of debwt_b200/synth.py generated in HBM (csrc/synth.cu), bit-identical to the numpy
generators.  torch only holds the device memory.  Bench / test plumbing, not part of the BWT path."""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from .binding import c_p, check, lib


def _u64(v):
    return ctypes.c_uint64(int(v) & ((1 << 64) - 1))


def _thr(rate: float) -> int:
    return int(rate * (1 << 53))


def random_bases(seed: int, n: int, device: int = 0) -> torch.Tensor:
    out = torch.empty(max(n, 1), dtype=torch.uint8, device=torch.device("cuda", device))
    check(lib().debwt_synth_random_bases(device, c_p(out.data_ptr()), _u64(n), _u64(seed)))
    return out[:n]


def genome_like(n: int, seed0: int, scale: float = 1.0, device: int = 0) -> torch.Tensor:
    """synth.genome_like on the device: iid background + three repeat families"""
    seq = random_bases(seed0, n, device)
    f = n / 3.1e9 * scale
    fams = [(seed0 + 1, int(1_000_000 * f), 300, 0.10), (seed0 + 2, int(100_000 * f), 6000, 0.03), (seed0 + 3, int(2_000 * f), 10_000, 0.0)]
    owner = None
    for seed, copies, length, rate in fams:
        if copies <= 0 or n <= length:
            continue
        if owner is None:
            owner = torch.zeros(n, dtype=torch.int32, device=seq.device)
        check(lib().debwt_synth_insert_family(device, c_p(seq.data_ptr()), _u64(n), _u64(seed), _u64(copies), _u64(length),
                                              _u64(_thr(rate)), c_p(owner.data_ptr())))
    del owner
    return seq


def mutate(seq: torch.Tensor, seed: int, rate: float) -> torch.Tensor:
    out = torch.empty_like(seq)
    check(lib().debwt_synth_mutate(seq.device.index or 0, c_p(seq.data_ptr()), c_p(out.data_ptr()), _u64(seq.numel()), _u64(seed),
                                   _u64(_thr(rate))))
    return out


def reverse_complement(seq: torch.Tensor) -> torch.Tensor:
    """the reverse complement of an upper-case ACGT sequence on the device (api.both_strands on the device)"""
    lut = torch.zeros(256, dtype=torch.uint8, device=seq.device)
    for x, y in (b"AT", b"CG", b"GC", b"TA"):
        lut[x] = y
    return lut[seq.long()].flip(0)


def join_records_device(records) -> tuple[torch.Tensor, np.ndarray]:
    """T = S1 # S2 # ... Sn $ in one device buffer + separator offsets (what api.join_records does on the host)"""
    n = sum(int(r.numel()) for r in records) + len(records)
    text = torch.empty(n, dtype=torch.uint8, device=records[0].device)
    seps = np.empty(len(records), dtype=np.uint64)
    pos = 0
    for i, r in enumerate(records):
        text[pos:pos + r.numel()] = r
        pos += int(r.numel())
        seps[i] = pos
        pos += 1
    text[torch.from_numpy(seps[:-1].astype(np.int64)).to(text.device)] = ord("#")
    text[-1] = ord("$")
    return text, seps


def config3(n: int = 3_100_000_000, n_records: int = 24, device: int = 0):
    """C3 (synth.config3): human-sized genome cut into n_records records; returns (device text, seps)"""
    seq = genome_like(n, 5, device=device)
    per = -(-n // n_records)
    return join_records_device([seq[i:i + per] for i in range(0, n, per)])


def config4(base_len: int = 300_000_000, n_genomes: int = 10, rate: float = 0.001, device: int = 0):
    """C4 (synth.config4): base genome + n_genomes-1 copies at `rate` substitution divergence"""
    base = genome_like(base_len, 9, device=device)
    return join_records_device([base] + [mutate(base, 10 + i, rate) for i in range(n_genomes - 1)])


def config2(n: int = 100_000_000, device: int = 0):
    """C2 has a host-side slot shuffle (argsort); generate with numpy and upload"""
    from . import api, synth
    text, seps = api.join_records(synth.config2(n))
    return torch.from_numpy(text).to(torch.device("cuda", device)), seps
