"""Bit-exact CPU model of the packed DP word (csrc/kernels_dp.cu, csrc/kernels_dpw.cu) on the library's own layout.

Both DP kernels keep a cell in one int32, score << S0 | q << (LB+XB) | x << LB | len, and make_dp_layout sizes the
fields from the scores.  A candidate below the score field wraps int32 into a high score, and an x or len that
outgrows its field carries into the fields above; either one changes results silently.  The full matrix and the
windows of the windowed path reach different ranges (a window that starts at column j0 > 1 starts from -inf in every
row), so both are modelled here, with the constants vfb_debug_dp_layout returns (the host code vfb_create runs):

  * the column loop of k2_dp_packed / k2_dp_window (the same loop: IMAD adds, VIADDMNMX, VIMNMX3, AND hmask), in
    int32 with wrap, rows padded to AMAX = A rounded up to 4 with wildcard rows, the last-row pick for A < AMAX, the
    `hA > bestcap` leftmost-best rule; each window from H = neg_e (column 0 when j0 = 1);
  * k2_dp_packed's end (last-column rule) and k2_resolve's key packing (DPW_BIAS, 0xFFFFF - j, the cb_val rule);
  * windows from a plain unit-cost edit-distance filter (test_window_model_cpu.py), [first - A - K, last].

and every read is checked for
  (a) no sum in rows 1..A leaves int32;
  (b) no x reaches 2^XB and no len 2^LB before it is incremented (nothing carries into q or the score);
  (c) the full kernel's (score, length) equals the oracle's;
  (d) the windowed path accepts exactly the reads the oracle accepts, with the oracle's (score, length).
Set VFB_SLOW_TESTS=1 for the long sweep of the whole scoring grid.
"""
import ctypes as C
import os
import random

import numpy as np
import pytest

import oracle
from oracle import twin
from vfind_b200 import api

from test_window_model_cpu import edit_distance_columns

slow = pytest.mark.skipif(os.environ.get("VFB_SLOW_TESTS") != "1", reason="long sweep: set VFB_SLOW_TESTS=1")

I32_LO, I32_HI = -(1 << 31), (1 << 31) - 1
INT_MIN_2 = -(1 << 30)            # INT_MIN / 2, the kernels' initial best
DPW_BIAS = 1 << 23
ADAPTER_LENS = [4, 5, 7, 8, 12, 13, 16, 18, 20, 21, 32, 33, 40, 47, 48, 64]
THRESHOLDS = [0.5, 0.6, 0.7, 0.75, 0.8, 0.9, 0.95]
# scorings whose windows wrapped int32 before the window range was part of the layout: (scoring, A, thr)
WRAPPED_BEFORE = [((2, -2, 5, 5), 20, 0.75), ((3, -3, 6, 6), 16, 0.8), ((10, -9, 7, 7), 12, 0.75),
                  ((4, -7, 10, 12), 32, 0.8), ((4, -7, 10, 12), 64, 0.8), ((1, -2, 3, 3), 12, 0.75),
                  ((1, -2, 3, 3), 24, 0.75), ((3, -2, 4, 4), 8, 0.75)]


class LayoutInfo(C.Structure):
    _fields_ = ([(n, C.c_int32) for n in ("packed", "max_edits", "accept_bound")] + [("lcap", C.c_uint32)] +
                [(n, C.c_int32) for n in ("S0", "LB", "XB", "c_eopen", "c_eext", "c_fopen", "c_fext", "hmask", "lowmask",
                                          "lenmask", "neg_e", "neg_f", "w_match", "w_mismatch", "w_wild")])


@pytest.fixture(scope="module")
def lib():
    L = api.load_library()
    L.vfb_debug_dp_layout.argtypes = [C.c_int32] * 4 + [C.c_uint32, C.c_double, C.c_int32, C.POINTER(LayoutInfo)]
    return L


def layout(lib, sc, A, thr, dp_mode=0):
    info = LayoutInfo()
    assert lib.vfb_debug_dp_layout(sc[0], sc[1], sc[2], sc[3], A, thr, dp_mode, C.byref(info)) == 0
    return {n: getattr(info, n) for n, _ in LayoutInfo._fields_}


def wrap(v):
    return ((v - I32_LO) & 0xFFFFFFFF) + I32_LO


def code(b):
    return {65: 0, 97: 0, 67: 1, 99: 1, 71: 2, 103: 2, 84: 3, 116: 3}.get(b, 4)      # dp_code


def run_columns(jobs):
    """The column loop of k2_dp_packed / k2_dp_window on a batch of jobs (layout, adapter, read, j0, j1) with adapters
    of one length, all lanes in lockstep as numpy int64 arrays holding int32 values.  Returns per job
    (best, bestj, H of column j1 rows 1..A, overflow, carry)."""
    A = len(jobs[0][1])
    AMAX = (A + 3) & ~3
    EXACT = A == AMAX
    n = len(jobs)

    def lane(key):
        return np.array([j[0][key] for j in jobs], dtype=np.int64)

    LB, XB = lane("LB"), lane("XB")
    lenmask, xmax = lane("lenmask"), (1 << XB) - 1
    c_eopen, c_eext, c_fopen, c_fext = lane("c_eopen"), lane("c_eext"), lane("c_fopen"), lane("c_fext")
    hmask, lowmask = lane("hmask"), lane("lowmask")
    # profile[c][i] per lane: rows past A and wildcards score 0; entry AMAX is what the last group's Wn (= W4) hands
    # row AMAX
    prof = np.empty((n, 5, AMAX + 1), dtype=np.int64)
    for w, (lay, ad, _, _, _) in enumerate(jobs):
        prof[w] = lay["w_wild"]
        for i in range(A):
            a = code(ad[i])
            for c in range(4):
                if a < 4:
                    prof[w, c, i] = lay["w_match"] if a == c else lay["w_mismatch"]
        prof[w, :, AMAX] = prof[w, :, AMAX - 4]
    j0 = np.array([j[3] for j in jobs])
    ncol = np.array([j[4] - j[3] + 1 for j in jobs])
    T = int(ncol.max())
    codes = np.full((T, n), 4, dtype=np.int64)
    for w, (_, _, read, a0, a1) in enumerate(jobs):
        codes[:a1 - a0 + 1, w] = [code(b) for b in read[a0 - 1:a1]]
    H = np.empty((AMAX, n), dtype=np.int64)
    H[:] = np.where(j0 == 1, 0, lane("neg_e"))             # column 0 is the true border; elsewhere -inf
    E = np.empty((AMAX, n), dtype=np.int64)
    E[:] = lane("neg_e")
    neg_f = lane("neg_f")
    best = np.full(n, INT_MIN_2, dtype=np.int64)
    bestcap = best.copy()
    bestj = np.zeros(n, dtype=np.int64)
    Hend = np.zeros((A, n), dtype=np.int64)
    over = np.zeros(n, dtype=bool)
    carry = np.zeros(n, dtype=bool)
    lanes = np.arange(n)

    for t in range(T):
        act = t < ncol
        W = prof[lanes, codes[t]].T                         # W[i]: row i's increment for each lane's byte
        hup = np.zeros(n, dtype=np.int64)
        F = neg_f.copy()
        d = W[0].copy()
        for i in range(AMAX):
            hl = H[i]
            dn = hl + W[i + 1]
            e_ext, e_open = E[i] + c_eext, hl + c_eopen
            f_ext, f_open = F + c_fext, hup + c_fopen
            if i < A:                                       # rows 1..A; dn feeds row i + 2
                lo = np.minimum(np.minimum(e_ext, e_open), np.minimum(f_ext, f_open))
                hi = np.maximum(np.maximum(e_ext, e_open), np.maximum(f_ext, f_open))
                if i + 1 < A:
                    lo, hi = np.minimum(lo, dn), np.maximum(hi, dn)
                over |= act & ((lo < I32_LO) | (hi > I32_HI))
                # each add sets len + 1, extensions also x + 1: the field must not be full already
                full = (((E[i] >> LB) & xmax) == xmax) | (((F >> LB) & xmax) == xmax)
                full |= ((E[i] & lenmask) == lenmask) | ((F & lenmask) == lenmask)
                full |= ((hl & lenmask) == lenmask) | ((hup & lenmask) == lenmask)
                carry |= act & full
            ee = np.maximum(wrap(e_open), wrap(e_ext))      # __viaddmax_s32(hl, c_eopen, E + c_eext)
            ff = np.maximum(wrap(f_open), wrap(f_ext))
            h = np.maximum(np.maximum(d, ff), ee) & hmask   # __vimax3_s32(d, ff, ee) & hmask
            E[i] = ee
            F = ff
            H[i] = h
            hup = h
            d = wrap(dn)
        hA = H[AMAX - 1]
        if not EXACT:
            if A == AMAX - 1:
                hA = H[AMAX - 2]
            if A == AMAX - 2:
                hA = H[AMAX - 3]
            if A == AMAX - 3:
                hA = H[AMAX - 4]
        upd = act & (hA > bestcap)
        best = np.where(upd, hA, best)
        bestcap = np.where(upd, hA | lowmask, bestcap)
        bestj = np.where(upd, j0 + t, bestj)
        last = ncol - 1 == t
        Hend[:, last] = H[:A, last]
    return [(int(best[w]), int(bestj[w]), [int(v) for v in Hend[:, w]], bool(over[w]), bool(carry[w])) for w in range(n)]


def last_column_best(lay, Hcol):
    cb, cbcap = INT_MIN_2, INT_MIN_2
    for h in Hcol:                                          # smallest row with the best score
        if h > cbcap:
            cb, cbcap = h, h | lay["lowmask"]
    return cb


def full_kernel_plan(lay, ad, reads):
    """k2_dp_packed: jobs, and what turns their results into (score, len, overflow, carry) per read."""
    S0 = lay["S0"]

    def finish(results):
        out = []
        for read, (best, bestj, Hcol, ov, ca) in zip(reads, results):
            cb = last_column_best(lay, Hcol)
            fin = best
            if (cb >> S0) > (best >> S0) or ((cb >> S0) == (best >> S0) and bestj == len(read)):
                fin = cb
            out.append((fin >> S0, fin & lay["lenmask"], ov, ca))
        return out
    return [(lay, ad, r, 1, len(r)) for r in reads], finish


def filter_windows(ad, read, K):
    """k2_filter's windows: groups of columns with ed <= K (a group closes at a gap > A + K), [first - A - K, last]."""
    A, L = len(ad), len(read)
    span = A + K
    ed = edit_distance_columns(ad, read)
    wins, first, last = [], 0, 0
    for j in range(1, L + 1):
        if ed[j] <= K:
            if first and j - last > span:
                wins.append((max(1, first - span), min(last, L)))
                first = 0
            if not first:
                first = j
            last = j
    if first:
        wins.append((max(1, first - span), min(last, L)))
    return wins


def windowed_plan(lay, K, ad, reads):
    """k2_filter -> k2_dp_window -> k2_resolve: jobs, and what turns their results into (score or None, len, overflow,
    carry) per read (None: no window, k2_resolve leaves the read alone)."""
    S0, lenmask = lay["S0"], lay["lenmask"]
    jobs, owner = [], []
    for r, read in enumerate(reads):
        for j0, j1 in filter_windows(ad, read, K):
            jobs.append((lay, ad, read, j0, j1))
            owner.append(r)

    def finish(results):
        best_key = [0] * len(reads)
        cb_val = [0] * len(reads)
        ov = [False] * len(reads)
        ca = [False] * len(reads)
        for (_, _, read, j0, j1), r, (best, bestj, Hcol, o, c) in zip(jobs, owner, results):
            key = ((best >> S0) + DPW_BIAS) << 40 | (0xFFFFF - bestj) << 20 | (best & lenmask)
            best_key[r] = max(best_key[r], key)             # atomicMax
            if j1 == len(read):
                cb = last_column_best(lay, Hcol)
                cb_val[r] = ((cb >> S0) + DPW_BIAS) << 32 | (cb & lenmask)
            ov[r] |= o
            ca[r] |= c
        out = []
        for r, read in enumerate(reads):
            key = best_key[r]
            if not key:
                out.append((None, None, ov[r], ca[r]))
                continue
            score = (key >> 40) - DPW_BIAS
            bestj = 0xFFFFF - ((key >> 20) & 0xFFFFF)
            ln = key & 0xFFFFF
            if cb_val[r]:
                cs = (cb_val[r] >> 32) - DPW_BIAS
                if cs > score or (cs == score and bestj == len(read)):
                    score, ln = cs, cb_val[r] & 0xFFFFFFFF
            out.append((score, ln, ov[r], ca[r]))
        return out
    return jobs, finish


def run_plans(plans):
    """Runs the jobs of several plans (adapters of one length) as one batch; each plan's finished results."""
    jobs = [j for p in plans for j in p[0]]
    results = run_columns(jobs) if jobs else []
    out, k = [], 0
    for p_jobs, finish in plans:
        out.append(finish(results[k:k + len(p_jobs)]))
        k += len(p_jobs)
    return out


# ------------------------------------------------------------------------------------ reads
def mutate(rng, ad, n_edits):
    m = bytearray(ad)
    for _ in range(n_edits):
        p = rng.randrange(len(m)) if m else 0
        op = rng.random()
        if op < 0.4 and m:
            m[p] = rng.choice(b"ACGT".replace(bytes([m[p]]), b"") or b"ACGT")
        elif op < 0.7 and len(m) > 1:
            del m[p]
        else:
            m.insert(p, rng.choice(b"ACGT"))
    return bytes(m)


def diagonal_junk(rng, ad, n):
    """n bases that mismatch the adapter on a few shifted diagonals: the cells under the -inf border of a window
    that starts in them stay on losing diagonal chains, as deep as the scores go."""
    A = len(ad)
    shifts = [rng.randrange(A) for _ in range(3)]
    out = bytearray()
    for p in range(n):
        avoid = {ad[(p + s) % A] for s in shifts}
        out.append(rng.choice([b for b in b"ACGT" if b not in avoid] or list(b"ACGT")))
    return bytes(out)


def adapters_for(rng, A):
    yield bytes(rng.choice(b"ACGT") for _ in range(A))
    yield (b"ACGT"[rng.randrange(4):][:1]) * A                                # homopolymer
    unit = bytes(rng.choice(b"ACGT") for _ in range(rng.choice((2, 3))))
    yield (unit * A)[:A]                                                       # repeat


def make_reads(rng, ad, K, n):
    A = len(ad)
    reads = []
    for it in range(n):
        kind = it % 4
        edits = rng.randint(0, K + 2)
        if kind == 0:       # junk on shifted diagonals over the A + K columns before a mutated adapter
            read = diagonal_junk(rng, ad, A + K + rng.randint(0, A)) + mutate(rng, ad, edits) + \
                bytes(rng.choice(b"ACGT") for _ in range(rng.randint(0, 8)))
        elif kind == 1:     # random junk, the adapter somewhere inside, maybe twice
            read = bytes(rng.choice(b"ACGT") for _ in range(rng.randint(A, 2 * A))) + mutate(rng, ad, edits)
            if rng.random() < 0.5:
                read += diagonal_junk(rng, ad, rng.randint(0, A)) + mutate(rng, ad, rng.randint(0, K + 2))
            read += bytes(rng.choice(b"ACGT") for _ in range(rng.randint(0, 12)))
        elif kind == 2:     # cut by the read's right end
            read = diagonal_junk(rng, ad, A + K + rng.randint(0, 8)) + mutate(rng, ad, edits)[:A - rng.randint(1, max(1, A // 4))]
        else:               # cut by the read's left end
            read = mutate(rng, ad, edits)[rng.randint(1, max(1, A // 4)):] + diagonal_junk(rng, ad, rng.randint(0, 2 * A))
        reads.append(read or b"A")
    return reads


# ------------------------------------------------------------------------------------ checks
def check_config(lib, sc, A, thr, n_reads, seed):
    """Runs (a)-(d) for one scoring / adapter length / threshold; returns the number of windowed reads checked."""
    lay0 = layout(lib, sc, A, thr, dp_mode=0)
    lay1 = layout(lib, sc, A, thr, dp_mode=1)
    assert lay0["packed"] == lay1["packed"] or (lay1["packed"] and lay0["max_edits"] < 0), (lay0, lay1)
    if not lay1["packed"]:
        return 0
    T, K = lay0["accept_bound"], lay0["max_edits"]
    for lay in (lay0, lay1):
        assert lay["S0"] == lay["LB"] + lay["XB"] + 2 and lay["lcap"] >= 1
        assert lay["lenmask"] == (1 << lay["LB"]) - 1 and lay["lowmask"] == (1 << lay["S0"]) - 1
    rng = random.Random(seed)
    cases, plans = [], []
    for ad in adapters_for(rng, A):
        reads = make_reads(rng, ad, max(K, 3), n_reads)
        want = [oracle.sg_stats(ad, r, *sc)[:2] for r in reads]
        for lay in [lay0] if lay0 == lay1 else [lay0, lay1]:    # fallback reads of the windowed path run on lay0
            cases.append(("full", ad, reads, want))
            plans.append(full_kernel_plan(lay, ad, reads))
        if K >= 0:
            cases.append(("window", ad, reads, want))
            plans.append(windowed_plan(lay0, K, ad, reads))
    checked = 0
    for (kind, ad, reads, want), got in zip(cases, run_plans(plans)):
        for r, w, (s, ln, ov, ca) in zip(reads, want, got):
            ctx = (kind, sc, A, thr, T, K, ad, r, (s, ln), w)
            if kind == "full":
                assert (s, ln) == w, ctx
            elif w[0] >= T:
                assert (s, ln) == w, ("accepted alignment differs",) + ctx
            else:
                assert s is None or s < T, ("rejected alignment accepted",) + ctx
            assert not ov, ("int32 overflow",) + ctx
            assert not ca, ("x / len field carry",) + ctx
            checked += kind == "window"
    return checked


def grid_sample(rng, n):
    out = []
    while len(out) < n:
        sc = (rng.randint(1, 10), -rng.randint(1, 10), rng.randint(0, 15), rng.randint(0, 15))
        out.append((sc, rng.choice(ADAPTER_LENS), rng.choice(THRESHOLDS)))
    return out


def test_layout_probe_matches_the_documented_defaults(lib):
    # C3: 20-base adapters at 0.75, windowed; one score bit more than the full kernel's layout (its windows start at
    # -inf and reach scores down to neg + (A-1)*wmin - o - e = -91), so the longest packed read is 2^16 - 1 - 20
    win, full = layout(lib, (3, -2, 5, 2), 20, 0.75), layout(lib, (3, -2, 5, 2), 20, 0.75, dp_mode=1)
    assert (win["packed"], win["max_edits"], win["accept_bound"]) == (1, 5, 46)
    assert (win["S0"], win["LB"], win["XB"], win["lcap"]) == (24, 16, 6, 65515)
    assert (full["packed"], full["max_edits"], full["S0"], full["LB"], full["XB"], full["lcap"]) == (1, -1, 25, 17, 6, 131051)
    assert full["neg_e"] == -46 << 25 and full["w_match"] == (3 << 25) + 1 + (2 << 23)
    # gaps that cost nothing: no window, and x needs as many bits as len
    z = layout(lib, (10, -10, 15, 0), 64, 0.75)
    assert z["packed"] and z["max_edits"] == -1 and z["lcap"] == (1 << z["XB"]) - 2
    assert layout(lib, (3, -2, 5, 2), 65, 0.75)["packed"] == 0                 # longer than the packed kernels take


@pytest.mark.parametrize("sc,A,thr", WRAPPED_BEFORE)
def test_windows_that_wrapped(lib, sc, A, thr):
    """The scorings whose windows wrapped int32 while the layout was sized for the full matrix only: gap costs above
    the mismatch cost, little headroom in the score field."""
    assert layout(lib, sc, A, thr)["max_edits"] >= 0, "these run the windowed path"
    assert check_config(lib, sc, A, thr, n_reads=160, seed=hash((sc, A, thr)) & 0xFFFF) > 0


def test_the_reported_read(lib):
    # adapter / read of the report: the oracle says (36, 20); a wrapped window said (63, 7), above the largest
    # possible score 40
    ad, read = b"TGGCCAGTAGATCTTCCCAA", b"ATAGCCTAGCTGGACATATTCACTTGGCCAGTAGATCTTCCCACCCGAAC"
    sc = (2, -2, 5, 5)
    lay = layout(lib, sc, 20, 0.75)
    assert twin.sg_stats(ad, read, *sc)[:2] == (36, 20)
    s, ln, ov, ca = run_plans([windowed_plan(lay, lay["max_edits"], ad, [read])])[0][0]
    assert (s, ln, ov, ca) == (36, 20, False, False)


@pytest.mark.parametrize("A", ADAPTER_LENS)
def test_every_instantiation(lib, A):
    # every AMAX and the row pick of A = AMAX - 1, - 2, - 3, under the defaults and under costly gaps
    for k, sc in enumerate([(3, -2, 5, 2), (2, -2, 5, 5), (1, -1, 4, 4)]):
        check_config(lib, sc, A, 0.8, n_reads=24, seed=100 * A + k)


def test_sampled_scoring_grid(lib):
    rng = random.Random(20261020)
    windowed = 0
    for k, (sc, A, thr) in enumerate(grid_sample(rng, 60)):
        windowed += check_config(lib, sc, A, thr, n_reads=16, seed=k) > 0
    assert windowed >= 8, windowed


@slow
def test_scoring_grid_long_sweep(lib):
    rng = random.Random(7)
    for k, (sc, A, thr) in enumerate(grid_sample(rng, 3000)):
        check_config(lib, sc, A, thr, n_reads=24, seed=k)
