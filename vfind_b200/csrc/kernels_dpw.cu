// K2 (windowed) — the same semi-global DP as kernels_dp.cu, restricted to the read columns where
// an ACCEPTED alignment can end, found first by a bit-parallel filter.  Results are identical
// to the full DP for every alignment the reference accepts (and every other one is rejected),
// see the argument below; what changes is the work: ~A+2K columns per read instead of all L.
//
// Why it is exact.  Let T be the integer accept bound (score >= T <=> score as f64 > min,
// /root/reference/src/lib.rs:157) and B = A*match - T the budget an accepted alignment may
// lose.  Every way of losing score is an "edit" with a positive cost: substitution
// (match - mismatch), wildcard column (match), adapter base left unaligned at a read end (match),
// inserted read base (open, then extend), skipped adapter base (match + open, then
// match + extend).  K = the largest number of edits whose cost fits in B (host, exact search).
//   (1) Filter: Myers' bit-vector algorithm gives, per column j, the unit-cost edit distance
//       ed(j) between the whole adapter and the best read substring ending at j (free start in
//       the read).  A path of the DP that ends at (A, j) with score >= T is an edit script with
//       at most K edits, so ed(j) <= K; a path ending at (i, L), i < A (adapter hanging over the
//       read end) gives ed(L) <= K as well, its unaligned tail counted as edits.  Columns with
//       ed(j) > K therefore cannot hold an accepted end cell.
//   (2) Window: a path with at most K edits that ends at column j starts no earlier than column
//       j - A - K.  The DP is run on [j - A - K, j] (merged over neighbouring flagged columns)
//       from the boundary H = -inf (H[0][.] = 0; the true border H[i][0] = 0 when the window
//       starts at column 1).  Boundary values are <= the true ones, so every computed value is
//       <= its true value; and a cell all of whose optimal paths lie inside the window — every
//       cell with true score >= T whose column is in the window's flagged part — has exactly its
//       true packed (score, length) value, because all candidates that tie for its maximum are
//       themselves ends of optimal sub-paths inside the window (induction on path length), so
//       the tie rules see the same candidates.
//   (3) End cell: the leftmost best last-row cell and the last-column rule only ever select a
//       cell with score >= T when the alignment is accepted; all such cells are exact, all other
//       cells are <= their true value < T.  If nothing reaches T the read is rejected, as in the
//       reference (its score is then not needed: only the accept decision reaches the table).
// The filter needs positive edit costs and a selective K (3K <= A); otherwise, for adapters longer than 64,
// and in diagnostics mode (exact scores of rejected alignments) the full kernel runs instead.  Adapters of up to 32
// bases use one 32-bit word per Myers vector, 33..64 bases one 64-bit word (two ALU instructions per logic op).
#include <climits>

#include "vfb_internal.cuh"

namespace vfb {

// ------------------------------------------------------------------------------------ host: K
int dpw_max_edits(const DpScoring &s, uint32_t A, int min_accept)
{
    // returns K >= 0, or -1 when the filter does not apply
    if (A < 4 || A > 64) return -1;
    if (s.match <= 0 || s.mismatch >= s.match || s.open <= 0 || s.extend <= 0) return -1;
    const long long B = (long long)A * s.match - min_accept;
    if (B < 0) return 0;                       // not even a perfect alignment reaches the bound
    const long long c_sub = (long long)s.match - s.mismatch;
    long long c1 = c_sub < s.match ? c_sub : s.match;          // substitution, wildcard, unaligned end
    if (c1 <= 0) return -1;
    long long best = 0;
    for (long long a = 0; a * s.open <= B; ++a) {
        for (long long b = 0; a * s.open + b * ((long long)s.match + s.open) <= B; ++b) {
            const long long rem = B - a * s.open - b * ((long long)s.match + s.open);
            long long cheapest = c1;
            if (a > 0 && s.extend < cheapest) cheapest = s.extend;
            if (b > 0 && s.match + s.extend < cheapest) cheapest = s.match + s.extend;
            const long long edits = a + b + rem / cheapest;
            if (edits > best) best = edits;
        }
    }
    if (best * 3 > (long long)A) return -1;    // not selective enough to pay for itself
    return (int)best;
}

// ------------------------------------------------------------------------------------ filter
#define DPW_THREADS 128
#define DPW_WARPS (DPW_THREADS / 32)
#define DPW_BIAS (1 << 23)

struct WinItem {
    uint32_t read, item, j0, j1;      // columns j0..j1 (1-based, inclusive) of read `read`
};

struct DpwArgs {
    DpJob job;
    DpLayout lay;
    int K;
    uint32_t lcap;
    WinItem *wins;
    uint32_t *n_wins;
    uint32_t win_cap;
    unsigned long long *best_key;     // per worklist item: (score+BIAS)<<40 | (0xFFFFF-j)<<20 | len
    unsigned long long *cb_val;       // per worklist item: (score+BIAS)<<32 | len, 0 = window did not reach column L
    uint32_t *fallback, *n_fallback;  // reads handed to the full kernel
    unsigned long long *cells_computed;
    uint32_t *work;                   // [32]: the window kernel's cursor (next unclaimed window; warps claim 32 at a time)
};

__device__ __forceinline__ void win_emit(const DpwArgs &a, uint32_t r, uint32_t item, int first, int last, int span, int L,
                                         bool &overflow)
{
    int j0 = first - span;
    if (j0 < 1) j0 = 1;
    const uint32_t p = atomicAdd(a.n_wins, 1u);
    if (p < a.win_cap) a.wins[p] = WinItem{r, item, (uint32_t)j0, (uint32_t)(last > L ? L : last)};
    else overflow = true;
}

// One column of Myers' bit-vector recurrence.  The adapter occupies the HIGH A bits of the word
// (row A = the top bit, so the score delta is the top bit of Ph / Mh); the low bits are rows
// that match every byte and start at D = 0, which leaves the adapter rows' values unchanged
// (a free text start already gives them D[0][j] = 0 underneath).
template <typename W>
__device__ __forceinline__ void myers_col(W Eq, W &Pv, W &Mv, int &score)
{
    constexpr int TOP = (int)sizeof(W) * 8 - 1;
    const W Xv = Eq | Mv;
    const W Xh = (((Eq & Pv) + Pv) ^ Pv) | Eq;
    W Ph = Mv | ~(Xh | Pv);
    W Mh = Pv & Xh;
    score += (int)(Ph >> TOP);
    score -= (int)(Mh >> TOP);
    Ph <<= 1;
    Mh <<= 1;
    Pv = Mh | ~(Xv | Ph);
    Mv = Ph & Xv;
}

// Filter: one lane = one read, streamed as 16-byte aligned chunks (LDG.128, next chunk prefetched).
// The <= 15 bytes of the first chunk that precede the read are run through the recurrence as
// well: extra text on the left can only lower ed(j), so the flagged set stays a superset.  Each
// chunk first runs 16 unrolled columns tracking only the minimum of ed; the (few) chunks whose
// minimum reaches K are replayed from the saved state with the per-column window bookkeeping.
// Byte -> Eq goes through a small table keyed by the byte's low bits (6 bits for 32-bit words, 5 bits for
// 64-bit words — the key times the entry size must fit a byte lane; entries OR-ed over the bytes that
// share a key: again a superset, and exact for every letter).
// Blocks per SM of the filter grid: many more blocks than fit at once, so the block scheduler evens out the cost of
// the items (see the loop below).  Filter time per 100 M reads on one B200 by blocks per SM: 12: 13.6 ms, 24: 12.9,
// 48: 12.6, 96: 12.5, 192: 12.7.
#define FILTER_BPS 48

template <typename W>
__global__ void __launch_bounds__(DPW_THREADS, sizeof(W) == 4 ? 8 : 5)
k2_filter(const __grid_constant__ DpwArgs a)
{
    constexpr int BITS = (int)sizeof(W) * 8;
    constexpr int KEYBITS = sizeof(W) == 4 ? 6 : 5;
    constexpr int ESH = sizeof(W) == 4 ? 2 : 3;               // log2(entry size)
    constexpr uint32_t KMASK = ((1u << KEYBITS) - 1u) * 0x01010101u;
    __shared__ W lutEq[1 << KEYBITS];
    const DpJob &job = a.job;
    const int A = (int)job.adapter_len;
    const int sh = BITS - A;
    if (threadIdx.x < (1 << KEYBITS)) {
        W m = sh ? (((W)1 << sh) - (W)1) : (W)0;
        for (int b = threadIdx.x; b < 256; b += (1 << KEYBITS)) {
            const int c = dp_code((uint8_t)b);
            if (c < 4)
                for (int i = 0; i < A; ++i)
                    if (job.adapter_code[i] == c) m |= (W)1 << (i + sh);
        }
        lutEq[threadIdx.x] = m;
    }
    __syncthreads();
    const unsigned char *lutb = reinterpret_cast<const unsigned char *>(lutEq);
    const int lane = threadIdx.x & 31;
    const uint32_t n_items = *job.n_items;
    const int span = A + a.K;
    const int K = a.K;
    unsigned long long cells = 0;
    // (a static grid-stride share per block, but many more blocks than fit at once: the block scheduler evens
    // out the differences in cost between items; claiming work from a global cursor, as k2_dp_window does, made
    // this kernel 3.5x slower)
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t base = blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < n_items; base += stride) {
        const uint32_t item = base + lane;
        if (item >= n_items) continue;
        const uint32_t r = job.worklist[item];
        const vfb_span sp = job.spans[r];
        const int L = (int)sp.len;
        if (L == 0) continue;
        if (sp.len > a.lcap || sp.len >= (1u << 20)) {
            a.fallback[atomicAdd(a.n_fallback, 1u)] = r;       // full kernel (it counts its own cells)
            continue;
        }
        const uintptr_t addr = reinterpret_cast<uintptr_t>(job.text + sp.off);
        const uint4 *base16 = reinterpret_cast<const uint4 *>(addr & ~(uintptr_t)15);
        const int lead = (int)(addr & 15u);
        const int n_chunks = (lead + L + 15) >> 4;
        W Pv = ~(W)0 << sh, Mv = 0;
        int score = A;
        int first = 0, last = 0;          // current group of flagged columns (0 = none)
        bool overflow = false;
        uint4 nx = __ldg(base16), nx2 = n_chunks > 1 ? __ldg(base16 + 1) : make_uint4(0, 0, 0, 0);
        for (int c = 0; c < n_chunks; ++c) {
            const uint4 v = nx;               // two chunks in flight
            nx = nx2;
            if (c + 2 < n_chunks) nx2 = __ldg(base16 + c + 2);
            const uint32_t w[4] = {v.x, v.y, v.z, v.w};
            const W Pv0 = Pv, Mv0 = Mv;
            const int score0 = score;
            int mn = INT_MAX;
#pragma unroll
            for (int wi = 0; wi < 4; ++wi) {
                const uint32_t w4 = (w[wi] & KMASK) << ESH;
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    const uint32_t key = __byte_perm(w4, 0, 0x4440 + b);
                    myers_col<W>(*reinterpret_cast<const W *>(lutb + key), Pv, Mv, score);
                    mn = min(mn, score);
                }
            }
            if (mn <= K) {
                // replay this chunk from the saved state, collecting the flagged columns
                Pv = Pv0; Mv = Mv0; score = score0;
                uint32_t flags = 0;
#pragma unroll
                for (int wi = 0; wi < 4; ++wi) {
                    const uint32_t w4 = (w[wi] & KMASK) << ESH;
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        const uint32_t key = __byte_perm(w4, 0, 0x4440 + b);
                        myers_col<W>(*reinterpret_cast<const W *>(lutb + key), Pv, Mv, score);
                        if (score <= K) flags |= 1u << (wi * 4 + b);
                    }
                }
                const int jbase = c * 16 - lead + 1;      // column (1-based) of the chunk's first byte
                while (flags) {
                    const int j = jbase + __ffs((int)flags) - 1;
                    flags &= flags - 1;
                    if (j < 1 || j > L) continue;
                    if (first && j - last > span) {             // far from the previous group: close it
                        win_emit(a, r, item, first, last, span, L, overflow);
                        first = 0;
                    }
                    if (!first) first = j;
                    last = j;
                }
            }
        }
        if (first) win_emit(a, r, item, first, last, span, L, overflow);
        if (overflow) {
            // the window list is full: the full kernel takes the whole read, and the poisoned key
            // makes k2_resolve skip whatever windows of it did get in
            a.best_key[item] = ~0ull;
            a.fallback[atomicAdd(a.n_fallback, 1u)] = r;
        } else {
            cells += (unsigned long long)L * (unsigned long long)A;     // (the full kernel counts its own)
        }
    }
    if (job.cells) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cells += __shfl_xor_sync(0xffffffffu, cells, o);
        if (lane == 0 && cells) atomicAdd(job.cells, cells);
    }
}

// ------------------------------------------------------------------------------------ window DP
// Same cell as k2_dp_packed (kernels_dp.cu): 3 IMAD + 2 VIADDMNMX + 1 VIMNMX3 + 1 LOP3.
template <int AMAX> struct DpwOcc { static constexpr int value = AMAX <= 20 ? 6 : (AMAX <= 28 ? 4 : (AMAX <= 40 ? 3 : 2)); };

template <int AMAX, bool EXACT>
__global__ void __launch_bounds__(DPW_THREADS, DpwOcc<AMAX>::value)
k2_dp_window(const __grid_constant__ DpwArgs a)
{
    constexpr int NG = AMAX / 4;
    extern __shared__ __align__(16) unsigned char smem[];
    int4 *prof = reinterpret_cast<int4 *>(smem);                 // [NG][8]
    uint8_t *lut = smem + NG * 8 * sizeof(int4);                 // byte -> 16 * code
    const DpJob &job = a.job;
    const DpLayout &lay = a.lay;
    const int A = (int)job.adapter_len;
    for (int idx = threadIdx.x; idx < NG * 8 * 4; idx += blockDim.x) {
        int g = idx >> 5, c = (idx >> 2) & 7, r = idx & 3, i = g * 4 + r;
        int w = lay.w_wild;
        if (i < A) {
            int ac = job.adapter_code[i];
            if (ac < 4 && c < 4) w = (ac == c) ? lay.w_match : lay.w_mismatch;
        }
        reinterpret_cast<int *>(prof)[idx] = w;
    }
    for (int idx = threadIdx.x; idx < 256; idx += blockDim.x) lut[idx] = (uint8_t)(16 * dp_code((uint8_t)idx));
    __syncthreads();

    const int lane = threadIdx.x & 31;
    uint32_t n_wins = *a.n_wins;
    if (n_wins > a.win_cap) n_wins = a.win_cap;
    const int c_eopen = lay.c_eopen, c_eext = lay.c_eext, c_fopen = lay.c_fopen, c_fext = lay.c_fext;
    const int hmask = lay.hmask, lowmask = lay.lowmask, one = lay.one;
    const int S0 = lay.S0;
    const unsigned char *profb = reinterpret_cast<const unsigned char *>(prof);
    unsigned long long cells = 0;

    for (;;) {
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(a.work + 32, 32u);
        base = __shfl_sync(0xffffffffu, base, 0);
        if (base >= n_wins) break;
        const uint32_t w = base + lane;
        const bool have = w < n_wins;
        WinItem it = have ? a.wins[w] : WinItem{0u, 0u, 1u, 0u};
        const vfb_span sp = have ? job.spans[it.read] : vfb_span{0u, 0u};
        const int L = (int)sp.len;
        const int j0 = (int)it.j0, j1 = have ? (int)it.j1 : 0;
        const uint8_t *seq = job.text + sp.off;
        int H[AMAX], E[AMAX];
        const int hinit = j0 == 1 ? 0 : lay.neg_e;      // column 0 is the true border; elsewhere -inf
#pragma unroll
        for (int i = 0; i < AMAX; ++i) { H[i] = hinit; E[i] = lay.neg_e; }
        int best = INT_MIN / 2, bestcap = INT_MIN / 2, bestj = 0;
        cells += (unsigned long long)(j1 >= j0 ? j1 - j0 + 1 : 0) * (unsigned long long)A;
        // the read's byte for column j+1 is fetched while column j is computed: the global load never
        // sits at the head of a column's dependency chain
        uint32_t bn = j1 >= j0 ? __ldg(seq + j0 - 1) : 0u;
        for (int j = j0; j <= j1; ++j) {
            const int c16 = lut[bn];
            if (j < j1) bn = __ldg(seq + j);
            const int4 *pc = reinterpret_cast<const int4 *>(profb + c16);
            int hup = 0, F = lay.neg_f;
            int4 W4 = pc[0];
            int d = W4.x;
#pragma unroll
            for (int gi = 0; gi < NG; ++gi) {
                int4 Wn = W4;
                if (gi + 1 < NG) Wn = pc[(gi + 1) * 8];
                const int Wv[5] = {W4.x, W4.y, W4.z, W4.w, Wn.x};
#pragma unroll
                for (int rI = 0; rI < 4; ++rI) {
                    const int i = gi * 4 + rI;
                    const int hl = H[i];
                    const int dn = hl * one + Wv[rI + 1];
                    int ee = E[i] * one + c_eext;
                    ee = __viaddmax_s32(hl, c_eopen, ee);
                    int ff = F * one + c_fext;
                    ff = __viaddmax_s32(hup, c_fopen, ff);
                    const int h = __vimax3_s32(d, ff, ee) & hmask;
                    E[i] = ee; F = ff; H[i] = h; hup = h; d = dn;
                }
                W4 = Wn;
            }
            int hA = H[AMAX - 1];
            if (!EXACT) {
                if (A == AMAX - 1) hA = H[AMAX - 2];
                if (A == AMAX - 2) hA = H[AMAX - 3];
                if (A == AMAX - 3) hA = H[AMAX - 4];
            }
            if (hA > bestcap) { best = hA; bestcap = hA | lowmask; bestj = j; }
        }
        if (have && j1 >= j0) {
            const long long bs = best >> S0;
            const unsigned long long key = ((unsigned long long)(bs + DPW_BIAS) << 40) |
                                           ((unsigned long long)(0xFFFFF - bestj) << 20) |
                                           (unsigned long long)(best & lay.lenmask);
            atomicMax(&a.best_key[it.item], key);
            if (j1 == L) {
                int cb = INT_MIN / 2, cbcap = INT_MIN / 2;
#pragma unroll
                for (int i = 0; i < AMAX; ++i)
                    if (i < A && H[i] > cbcap) { cb = H[i]; cbcap = H[i] | lowmask; }
                const long long cs = cb >> S0;
                a.cb_val[it.item] = ((unsigned long long)(cs + DPW_BIAS) << 32) | (unsigned long long)(cb & lay.lenmask);
            }
        }
    }
    if (a.cells_computed) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cells += __shfl_xor_sync(0xffffffffu, cells, o);
        if (lane == 0 && cells) atomicAdd(a.cells_computed, cells);
    }
}

// ------------------------------------------------------------------------------------ resolve
__global__ void __launch_bounds__(256)
k2_resolve(const __grid_constant__ DpwArgs a)
{
    const DpJob &job = a.job;
    const uint32_t n_items = *job.n_items;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    bool want_next = false;
    uint32_t r = 0;
    if (i < n_items) {
        const unsigned long long key = a.best_key[i];
        if (key && key != ~0ull) {
            r = job.worklist[i];
            const int L = (int)job.spans[r].len;
            int score = (int)(key >> 40) - DPW_BIAS;
            const int bestj = 0xFFFFF - (int)((key >> 20) & 0xFFFFFu);
            int len = (int)(key & 0xFFFFFu);
            const unsigned long long cbv = a.cb_val[i];
            if (cbv) {
                // last column replaces the last-row winner iff strictly better, or equal while the
                // row winner is the corner cell
                const int cs = (int)(cbv >> 32) - DPW_BIAS;
                if (cs > score || (cs == score && bestj == L)) { score = cs; len = (int)(cbv & 0xFFFFFFFFu); }
            }
            if (job.diag_score) { job.diag_score[r] = score; job.diag_len[r] = len; }
            if (score >= job.min_accept) {
                if (job.is_prefix) job.bound[r] = (uint32_t)len;
                else if (len <= L) job.bound[r] = (uint32_t)(L - len);
                want_next = job.next_list != nullptr && job.other_bound[r] == VFB_NONE;
            }
        }
    }
    if (job.next_list) {
        const unsigned m = __ballot_sync(0xffffffffu, want_next);
        if (m) {
            uint32_t base = 0;
            if (lane == 0) base = atomicAdd(job.n_next, (uint32_t)__popc(m));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (want_next) job.next_list[base + __popc(m & ((1u << lane) - 1))] = r;
        }
    }
}

template <int AMAX>
static int launch_window(const DpwArgs &args, int sm_count, cudaStream_t st)
{
    const bool exact = (int)args.job.adapter_len == AMAX;
    auto kern = exact ? k2_dp_window<AMAX, true> : k2_dp_window<AMAX, false>;
    const size_t smem = (AMAX / 4) * 8 * sizeof(int4) + 256;
    static int blocks_per_sm[2] = {0, 0};
    int &bps = blocks_per_sm[exact ? 1 : 0];
    if (!bps) {
        VFB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, DPW_THREADS, smem));
        if (bps < 1) bps = 1;
    }
    kern<<<sm_count * bps, DPW_THREADS, smem, st>>>(args);
    ++g_launches;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

int launch_dp_windowed(const DpJob &job, const DpLayout &lay, int K, uint32_t lcap, uint32_t max_items,
                       void *wins, uint32_t *n_wins, uint32_t win_cap, unsigned long long *best_key,
                       unsigned long long *cb_val, uint32_t *fallback, uint32_t *n_fallback,
                       unsigned long long *cells_computed, uint32_t *work_cursors, int sm_count, cudaStream_t st,
                       cudaEvent_t ev_filter_done, cudaEvent_t ev_windows_done)
{
    DpwArgs a;
    a.job = job; a.lay = lay; a.K = K; a.lcap = lcap;
    a.wins = static_cast<WinItem *>(wins); a.n_wins = n_wins; a.win_cap = win_cap;
    a.best_key = best_key; a.cb_val = cb_val; a.fallback = fallback; a.n_fallback = n_fallback;
    a.cells_computed = cells_computed;
    a.work = work_cursors;
    VFB_CUDA(cudaMemsetAsync(best_key, 0, (size_t)max_items * 8, st));
    VFB_CUDA(cudaMemsetAsync(cb_val, 0, (size_t)max_items * 8, st));
    if (job.adapter_len <= 32) k2_filter<uint32_t><<<sm_count * FILTER_BPS, DPW_THREADS, 0, st>>>(a);
    else k2_filter<unsigned long long><<<sm_count * FILTER_BPS, DPW_THREADS, 0, st>>>(a);
    ++g_launches;
    if (ev_filter_done) VFB_CUDA(cudaEventRecord(ev_filter_done, st));
    int rc;
    switch (((int)job.adapter_len + 3) & ~3) {
    case 4: rc = launch_window<4>(a, sm_count, st); break;
    case 8: rc = launch_window<8>(a, sm_count, st); break;
    case 12: rc = launch_window<12>(a, sm_count, st); break;
    case 16: rc = launch_window<16>(a, sm_count, st); break;
    case 20: rc = launch_window<20>(a, sm_count, st); break;
    case 24: rc = launch_window<24>(a, sm_count, st); break;
    case 28: rc = launch_window<28>(a, sm_count, st); break;
    case 32: rc = launch_window<32>(a, sm_count, st); break;
    case 36: rc = launch_window<36>(a, sm_count, st); break;
    case 40: rc = launch_window<40>(a, sm_count, st); break;
    case 44: rc = launch_window<44>(a, sm_count, st); break;
    case 48: rc = launch_window<48>(a, sm_count, st); break;
    case 52: rc = launch_window<52>(a, sm_count, st); break;
    case 56: rc = launch_window<56>(a, sm_count, st); break;
    case 60: rc = launch_window<60>(a, sm_count, st); break;
    case 64: rc = launch_window<64>(a, sm_count, st); break;
    default: set_error("adapter too long for the windowed DP"); return VFB_ERR_ARG;
    }
    if (rc) return rc;
    if (ev_windows_done) VFB_CUDA(cudaEventRecord(ev_windows_done, st));
    k2_resolve<<<(max_items + 255) / 256, 256, 0, st>>>(a);
    ++g_launches;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

uint32_t dpw_item_bytes() { return (uint32_t)sizeof(WinItem); }

}  // namespace vfb
