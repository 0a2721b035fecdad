"""both_strands in terms of the CPU oracle: the reverse complement and the two-pass composition the GPU must match.

Test infrastructure, like the oracle it composes (oracle.process_reads is run unchanged on the forward reads, then on
the reverse complements of the reads that have no region)."""
import numpy as np

from oracle import DIAG_DTYPE, INT32_MIN, Params, process_reads

_RC_LUT = np.arange(256, dtype=np.uint8)
_RC_LUT[np.frombuffer(b"ACGTUacgtu", dtype=np.uint8)] = np.frombuffer(b"TGCAAtgcaa", dtype=np.uint8)


def revcomp(seq: bytes) -> bytes:
    """Reverse complement: A<->T, C<->G, a<->t, c<->g, U->A, u->a; every other byte unchanged."""
    return _RC_LUT[np.frombuffer(bytes(seq), dtype=np.uint8)[::-1]].tobytes()


def has_region(diag, length):
    """The per-read predicate of a region (start, end located, start < end <= len): vfind_oracle.c do_read."""
    s, e = diag["start"].astype(np.int64), diag["end"].astype(np.int64)
    return (s >= 0) & (e >= 0) & (s < e) & (e <= np.asarray(length, dtype=np.int64))


def process_reads_both_strands(params: Params, text, off, length, n_threads=1, want_diag=False):
    """process_reads, then process_reads once more over the reverse complements of the reads that have no region
    (has_region) and are not empty; both count into one table.  A read counts on at most one strand.

    Returns (table dict, forward diag | None, reverse diag | None, cells of both passes).  The reverse diag has one
    row per read in read order: the reverse pass's values for the reads that were retried, the "absent" markers
    (-1, INT32_MIN for scores) elsewhere."""
    text = np.frombuffer(text, dtype=np.uint8) if isinstance(text, (bytes, bytearray)) else \
        np.ascontiguousarray(text, dtype=np.uint8)
    off = np.ascontiguousarray(off, dtype=np.uint32)
    length = np.ascontiguousarray(length, dtype=np.uint32)
    table, fdiag, cells = process_reads(params, text, off, length, n_threads=n_threads, want_diag=True)
    retry = np.nonzero(~has_region(fdiag, length) & (length > 0))[0]
    rlen = length[retry].astype(np.int64)
    roff = np.zeros(len(retry), dtype=np.int64)
    if len(retry):
        roff[1:] = np.cumsum(rlen[:-1])
    # gathered byte g of retried read i (at roff[i]) is the complement of text[off + len - 1 - (g - roff[i])]
    src = np.repeat(off[retry].astype(np.int64) + rlen - 1 + roff, rlen) - np.arange(int(rlen.sum()), dtype=np.int64)
    rtext = _RC_LUT[text[src]]
    rtable, rdiag_c, rcells = process_reads(params, rtext, roff.astype(np.uint32), rlen.astype(np.uint32),
                                            n_threads=n_threads, want_diag=want_diag)
    for k, v in rtable.items():
        table[k] = table.get(k, 0) + v
    rdiag = None
    if want_diag:
        rdiag = np.zeros(len(off), dtype=DIAG_DTYPE)
        for f in DIAG_DTYPE.names:
            rdiag[f] = INT32_MIN if f.startswith("score") else -1
        rdiag[retry] = rdiag_c
    return table, (fdiag if want_diag else None), rdiag, cells + rcells
