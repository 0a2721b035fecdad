"""umi_length in terms of the CPU oracle: the (variant, count, molecules) table the GPU must return.

Test infrastructure, like the oracles it composes: oracle.process_reads (and, for both_strands,
strand_oracle.process_reads_both_strands) decide every read's region; the key is formed from it as the C oracle does
(oracle.translate, or the bytes when they are UTF-8 under skip_translation), and the UMI is sliced from the read in the
orientation its region was found in."""
import numpy as np

import oracle
import strand_oracle


def process_reads_umi(params, text, off, length, umi_length, umi_offset=0, both_strands=False, n_threads=1):
    """Returns ({key: (count, molecules)}, reads_short, pairs).  pairs: distinct (key, UMI) pairs."""
    text = np.frombuffer(text, dtype=np.uint8) if isinstance(text, (bytes, bytearray)) else \
        np.ascontiguousarray(text, dtype=np.uint8)
    off = np.ascontiguousarray(off, dtype=np.uint32)
    length = np.ascontiguousarray(length, dtype=np.uint32)
    if both_strands:
        table, fdiag, rdiag, _ = strand_oracle.process_reads_both_strands(params, text, off, length, n_threads, True)
    else:
        table, fdiag, _ = oracle.process_reads(params, text, off, length, n_threads=n_threads, want_diag=True)
        rdiag = None
    fwd = strand_oracle.has_region(fdiag, length)
    rev = strand_oracle.has_region(rdiag, length) & ~fwd if rdiag is not None else np.zeros(len(off), dtype=bool)
    raw = text.tobytes()
    pairs = {}
    counted = {}
    short = 0
    for i in np.nonzero(fwd | rev)[0]:
        read = raw[int(off[i]):int(off[i]) + int(length[i])]
        d = fdiag[i] if fwd[i] else rdiag[i]
        if not fwd[i]:
            read = strand_oracle.revcomp(read)
        region = read[int(d["start"]):int(d["end"])]
        if params.skip_translation:
            key = region if oracle.is_utf8(region) else None
        else:
            key = oracle.translate(region)
        if key is None:
            continue
        counted[key] = counted.get(key, 0) + 1
        if len(read) < umi_offset + umi_length:
            short += 1
            continue
        umi = read[umi_offset:umi_offset + umi_length]
        pairs[(key, umi)] = pairs.get((key, umi), 0) + 1
    # self-check: the keys formed here are the ones the oracle counted
    assert counted == table, "umi oracle: keys differ from process_reads' table"
    out = {}
    for (key, _umi), c in pairs.items():
        cnt, mol = out.get(key, (0, 0))
        out[key] = (cnt + c, mol + 1)
    return out, short, len(pairs)


def umi_reads(seqs, params, umi_length, umi_offset=0, both_strands=False):
    """process_reads_umi over a list of byte strings."""
    text, off, ln = oracle.pack_reads(seqs)
    return process_reads_umi(params, text, off, ln, umi_length, umi_offset, both_strands)
