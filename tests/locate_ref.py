"""Reference suffix array for the locate tests, from the oracle's BWT (oracle/bwt_oracle.c, pinned on the reference's
golden vectors) inverted by a sequential LF walk on the CPU.  Independent of the CUDA path."""
import numpy as np

from oracle import coracle


def suffix_array_from_bwt(bwt_sym: np.ndarray) -> np.ndarray:
    """SA[row] = start position of the row's suffix, from BWT symbols (0..3, 4 '#', 5 '$').  All '#' are one symbol, so
    LF is the ordinary LF mapping over the 6-letter alphabet: LF(row of suffix i) = row of suffix i - 1."""
    b = np.ascontiguousarray(bwt_sym, dtype=np.uint8)
    n = b.size
    lf = np.empty(n, dtype=np.int64)
    lf[np.argsort(b, kind="stable")] = np.arange(n)
    lf = lf.tolist()
    sa = [0] * n
    r = int(np.flatnonzero(b == 5)[0])                   # the row of suffix 0 holds T[N-1] = '$'
    for pos in range(n):                                 # suffix 0, N-1, N-2, ..., 1
        sa[r] = (n - pos) % n
        r = lf[r]
    if r != int(np.flatnonzero(b == 5)[0]):
        raise ValueError("LF is not one N-cycle: not a BWT")
    return np.array(sa, dtype=np.uint64)


def suffix_array(sym: np.ndarray) -> np.ndarray:
    """SA of the text given as symbol codes (0..3, 4 '#', 5 '$'; '$' last), in the reference's suffix order"""
    return suffix_array_from_bwt(coracle.bwt_symbols(sym))
