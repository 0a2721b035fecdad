// K2 — batched inter-sequence semi-global affine-gap DP with the alignment-length statistic.
//
// Replaces `aligner.align(None, seq)` + get_score + get_length + the accept test of
// /root/reference/src/lib.rs:155-160 (parasail sg_stats_scan_profile_sat) for the reads whose
// adapter was not found exactly.  Rule set: SURVEY.md §8(c) (restated in DESIGN.md).
//
// Mapping: one lane = one alignment.  The adapter (rows, <= 64) lives in registers as two
// packed words per row (H and E of the previous column); the read (columns) streams through
// a per-warp shared-memory tile, transposed so that lane t reads bank t.  The adapter profile
// (packed diagonal increments per read-base code) sits in shared memory and is fetched four
// rows at a time with one conflict-free LDS.128.  Per cell: 3 adds (kept on the FMA pipe as
// IMAD), 2 VIADDMNMX, 1 VIMNMX3, 1 LOP3 — see DpLayout for how one max carries the length.
#include <climits>

#include "vfb_internal.cuh"

namespace vfb {

static inline int bits_for(uint64_t v)   // smallest b with 2^b > v
{
    int b = 0;
    while ((1ull << b) <= v) ++b;
    return b;
}

// The signed score field must hold every candidate any cell forms in rows 1..A, or an add wraps int32 and a low
// candidate turns into a high score.  Upper end: H <= smax = A*wmax.  Lower end (wmin <= 0 the cheapest step):
//   Full matrix: every H >= A*wmin (its diagonal runs back to row 0 or column 0, both 0), so H - o > neg; E and F
//   are >= neg (their border), and the lowest candidate is an extension of that border: >= neg - e (the bound
//   below takes neg - max(o, e)).
//   Window from column j0 > 1 (kernels_dpw.cu): H = neg in every row of column j0 - 1.  A cell (i, j) with
//   j - j0 + 1 < i has a diagonal that runs back into that border, so only H >= neg + (i-1)*wmin holds there; E and
//   F are >= that H - o, and an extension of them loses e more:  lowest >= neg + (A-1)*wmin - o - e.
//   Cells with j - j0 + 1 >= i reach row 0 on their diagonal and keep the full matrix's H >= i*wmin.
// x (an E run of extensions, which beats an opening at equal score) needs no more room in a window: a run whose
// last step is compared against an H past the triangle above (H >= i*wmin) loses at most smax - smin, as in the
// full matrix, and a run that ends inside the triangle has at most i <= A columns.
bool make_dp_layout(const DpScoring &s, uint32_t A, bool windowed, DpLayout *out)
{
    if (A < 1 || A > VFB_MAX_PACKED_ADAPTER) return false;
    if (s.open < 0 || s.extend < 0) return false;
    long long wmin = 0, wmax = 0;
    if (s.match < wmin) wmin = s.match;
    if (s.mismatch < wmin) wmin = s.mismatch;
    if (s.match > wmax) wmax = s.match;
    if (s.mismatch > wmax) wmax = s.mismatch;
    long long smax = (long long)A * wmax, smin = (long long)A * wmin;
    long long neg = smin - s.open - 1;           // border "-inf": below every real candidate
    long long lowest = neg - (s.open > s.extend ? s.open : s.extend);   // the lowest value ever formed (see above)
    if (windowed) lowest = neg + ((long long)A - 1) * wmin - s.open - s.extend;
    long long need = smax + 1 > -lowest ? smax + 1 : -lowest;
    if (need > (1 << 20)) return false;
    int SB = bits_for((uint64_t)need) + 1;       // signed field holding [-need, need]
    int budget = 30 - SB;                        // bits left for len + x
    if (budget < 10) return false;
    int LB, XB;
    int xbF = bits_for(A + 1);
    if (s.extend > 0) {
        long long xe = (smax - smin) / s.extend + 2;
        XB = bits_for((uint64_t)xe);
        if (XB < xbF) XB = xbF;
        LB = budget - XB;
        if (LB > 20) LB = 20;
    } else {
        // an extension run can be as long as the read: x needs as many bits as len
        LB = (budget + 1) / 2;
        XB = budget - LB;
        if (XB < xbF) return false;
        if (LB > 20) LB = 20;
    }
    if (LB < 7) return false;
    // longest read: len <= A + L < 2^LB, and with extend == 0 also L + 1 < 2^XB
    long long lcap = (1ll << LB) - 1 - A;
    if (s.extend == 0) {
        long long lx = (1ll << XB) - 2;
        if (lx < lcap) lcap = lx;
    }
    if (lcap < 1) return false;
    DpLayout L;
    L.LB = LB; L.XB = XB; L.S0 = LB + XB + 2;
    const int S0 = L.S0;
    const int X1 = 1 << LB, Q1 = 1 << (LB + XB), Q2 = 2 << (LB + XB);
    L.c_eopen = -s.open * (1 << S0) + 1;
    L.c_eext = -s.extend * (1 << S0) + 1 + X1;
    L.c_fopen = -s.open * (1 << S0) + 1 + Q1;
    L.c_fext = -s.extend * (1 << S0) + 1 + X1;
    L.hmask = ~(((1 << (XB + 2)) - 1) << LB);
    L.lowmask = (1 << S0) - 1;
    L.lenmask = (1 << LB) - 1;
    L.neg_e = (int)(neg * (1ll << S0));
    L.neg_f = (int)(neg * (1ll << S0)) + Q1;
    L.w_match = s.match * (1 << S0) + 1 + Q2;
    L.w_mismatch = s.mismatch * (1 << S0) + 1 + Q2;
    L.w_wild = 0 * (1 << S0) + 1 + Q2;
    L.one = 1;
    *out = L;
    return true;
}

__host__ __device__ static inline uint32_t dp_layout_lcap(const DpLayout &l, uint32_t A, int extend)
{
    long long lcap = (1ll << l.LB) - 1 - (long long)A;
    if (extend == 0) {
        long long lx = (1ll << l.XB) - 2;
        if (lx < lcap) lcap = lx;
    }
    return lcap < 0 ? 0u : (uint32_t)lcap;
}

#define DP_WARPS 4
#define DP_THREADS (DP_WARPS * 32)
#define DP_ROW 80   // bytes of ring buffer per lane: 4 slots x 16 B + 16 B pad (odd multiple of 16: no STS.128 conflicts beyond the 4-wavefront minimum)

struct DpKernelArgs {
    DpJob job;
    DpLayout lay;
    uint32_t lcap;          // longest read the packed layout can take
    uint32_t *fallback;     // worklist of items the packed kernel refused (nullable)
    uint32_t *n_fallback;
};

// Resident CTAs per SM the register budget is tuned for.
template <int AMAX> struct DpOcc { static constexpr int value = AMAX <= 20 ? 6 : (AMAX <= 28 ? 4 : (AMAX <= 44 ? 3 : 2)); };

template <int AMAX, bool EXACT>
__global__ void __launch_bounds__(DP_THREADS, DpOcc<AMAX>::value)
k2_dp_packed(const __grid_constant__ DpKernelArgs args)
{
    constexpr int NG = AMAX / 4;
    constexpr bool USE_IMAD = true;     // adds as IMAD (x*1+c): they issue on the FMA pipe, not the ALU pipe
    extern __shared__ __align__(16) unsigned char smem[];
    int4 *prof = reinterpret_cast<int4 *>(smem);                 // [NG][8] : rows 4g..4g+3 at code c
    uint8_t *lut = smem + NG * 8 * sizeof(int4);                 // byte -> 16 * code
    uint8_t *rings = lut + 256;                                  // [warp][lane][DP_ROW]

    const DpJob &job = args.job;
    const DpLayout &lay = args.lay;
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

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t *ring = rings + (warp * 32 + lane) * DP_ROW;         // private to this lane
    const uint32_t n_items = *job.n_items;
    const uint32_t n_groups = (n_items + 31) / 32;
    const uint32_t warps_total = gridDim.x * DP_WARPS;

    const int c_eopen = lay.c_eopen, c_eext = lay.c_eext, c_fopen = lay.c_fopen, c_fext = lay.c_fext;
    const int hmask = lay.hmask, lowmask = lay.lowmask, one = lay.one;
    const int S0 = lay.S0;
    const unsigned char *profb = reinterpret_cast<const unsigned char *>(prof);

    for (uint32_t g = blockIdx.x * DP_WARPS + warp; g < n_groups; g += warps_total) {
        const uint32_t item = g * 32 + lane;
        const bool have = item < n_items;
        const uint32_t r = have ? job.worklist[item] : 0u;
        vfb_span sp = have ? job.spans[r] : vfb_span{0u, 0u};
        bool run = have && sp.len > 0;
        if (run && sp.len > args.lcap) {
            // too long for the packed word: hand to the fallback kernel
            if (args.fallback) args.fallback[atomicAdd(args.n_fallback, 1u)] = r;
            run = false;
        }
        const int L = run ? (int)sp.len : 0;
        const int Lmax = __reduce_max_sync(0xffffffffu, L);
        if (job.cells) {
            unsigned long long c = (unsigned long long)L * (unsigned long long)A;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
            if (lane == 0 && c) atomicAdd(job.cells, c);
        }

        // The read streams through the lane's own ring: 16-byte aligned chunks, chunk m+2 is
        // in flight (registers) while the 16 columns of block m are computed.
        const uintptr_t addr = reinterpret_cast<uintptr_t>(job.text + sp.off);
        const uint4 *base16 = reinterpret_cast<const uint4 *>(addr & ~(uintptr_t)15);
        const int lead = (int)(addr & 15u);
        const int nch = L ? (lead + L + 15) >> 4 : 0;
        const uint4 z4 = make_uint4(0, 0, 0, 0);
        *reinterpret_cast<uint4 *>(ring) = nch > 0 ? __ldg(base16) : z4;
        *reinterpret_cast<uint4 *>(ring + 16) = nch > 1 ? __ldg(base16 + 1) : z4;
        uint4 nxt = nch > 2 ? __ldg(base16 + 2) : z4;

        int H[AMAX], E[AMAX];
#pragma unroll
        for (int i = 0; i < AMAX; ++i) { H[i] = 0; E[i] = lay.neg_e; }
        int best = INT_MIN / 2, bestcap = INT_MIN / 2, bestj = 0;

        for (int m = 0; m * 16 < Lmax; ++m) {
            const int kend = min(16, L - m * 16);
#pragma unroll 1
            for (int k = 0; k < kend; ++k) {
                const int c16 = lut[ring[(lead + m * 16 + k) & 63]];
                const int4 *pc = reinterpret_cast<const int4 *>(profb + c16);
                int hup = 0;                // H[0][j]   = 0
                int F = lay.neg_f;
                int4 W4 = pc[0];
                int d = W4.x;               // row 1 diagonal: H[0][j-1] + W = W
#pragma unroll
                for (int gi = 0; gi < NG; ++gi) {
                    int4 Wn = W4;
                    if (gi + 1 < NG) Wn = pc[(gi + 1) * 8];
                    const int Wv[5] = {W4.x, W4.y, W4.z, W4.w, Wn.x};
#pragma unroll
                    for (int rI = 0; rI < 4; ++rI) {
                        const int i = gi * 4 + rI;
                        const int hl = H[i];
                        // next row's diagonal candidate, taken before H[i] is overwritten
                        const int dn = USE_IMAD ? hl * one + Wv[rI + 1] : hl + Wv[rI + 1];
                        int ee = USE_IMAD ? E[i] * one + c_eext : E[i] + c_eext;
                        ee = __viaddmax_s32(hl, c_eopen, ee);
                        int ff = USE_IMAD ? F * one + c_fext : F + c_fext;
                        ff = __viaddmax_s32(hup, c_fopen, ff);
                        const int h = __vimax3_s32(d, ff, ee) & hmask;
                        E[i] = ee; F = ff; H[i] = h; hup = h; d = dn;
                    }
                    W4 = Wn;
                }
                // last row (row A, which is one of the four bottom register rows)
                int hA = H[AMAX - 1];
                if (!EXACT) {
                    if (A == AMAX - 1) hA = H[AMAX - 2];
                    if (A == AMAX - 2) hA = H[AMAX - 3];
                    if (A == AMAX - 3) hA = H[AMAX - 4];
                }
                if (hA > bestcap) { best = hA; bestcap = hA | lowmask; bestj = m * 16 + k + 1; }
            }
            // chunk m+2 lands in the ring, chunk m+3 takes off
            *reinterpret_cast<uint4 *>(ring + (((m + 2) & 3) << 4)) = nxt;
            nxt = m + 3 < nch ? __ldg(base16 + m + 3) : z4;
        }

        bool want_next = false;
        if (run) {
            // last column: smallest i with the best score
            int cb = INT_MIN / 2, cbcap = INT_MIN / 2;
#pragma unroll
            for (int i = 0; i < AMAX; ++i) {
                if (i < A && H[i] > cbcap) { cb = H[i]; cbcap = H[i] | lowmask; }
            }
            const int bs = best >> S0, cs = cb >> S0;
            int fin = best;
            if (cs > bs || (cs == bs && bestj == L)) fin = cb;
            const int score = fin >> S0, len = fin & lay.lenmask;
            if (job.diag_score) { job.diag_score[r] = score; job.diag_len[r] = len; }
            if (score >= job.min_accept) {
                if (job.is_prefix) job.bound[r] = (uint32_t)len;
                else if (len <= L) job.bound[r] = (uint32_t)(L - len);
                want_next = job.next_list != nullptr && job.other_bound[r] == VFB_NONE;
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
}

template <int AMAX>
static int launch_one(const DpKernelArgs &args, int sm_count, cudaStream_t st)
{
    const bool exact = (int)args.job.adapter_len == AMAX;
    auto kern = exact ? k2_dp_packed<AMAX, true> : k2_dp_packed<AMAX, false>;
    size_t smem = (AMAX / 4) * 8 * sizeof(int4) + 256 + DP_WARPS * 32 * DP_ROW;
    static int blocks_per_sm[2] = {0, 0};
    int &bps = blocks_per_sm[exact ? 1 : 0];
    if (!bps) {
        VFB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kern, DP_THREADS, smem));
        if (bps < 1) bps = 1;
    }
    kern<<<sm_count * bps, DP_THREADS, smem, st>>>(args);
    ++g_launches;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

int launch_dp_packed_ex(const DpJob &job, const DpLayout &lay, uint32_t lcap, uint32_t *fallback,
                        uint32_t *n_fallback, int sm_count, cudaStream_t st)
{
    DpKernelArgs args;
    args.job = job;
    args.lay = lay;
    args.lcap = lcap;
    args.fallback = fallback;
    args.n_fallback = n_fallback;
    const int A = (int)job.adapter_len;
    const int amax = (A + 3) & ~3;
    switch (amax) {
    case 4: return launch_one<4>(args, sm_count, st);
    case 8: return launch_one<8>(args, sm_count, st);
    case 12: return launch_one<12>(args, sm_count, st);
    case 16: return launch_one<16>(args, sm_count, st);
    case 20: return launch_one<20>(args, sm_count, st);
    case 24: return launch_one<24>(args, sm_count, st);
    case 28: return launch_one<28>(args, sm_count, st);
    case 32: return launch_one<32>(args, sm_count, st);
    case 36: return launch_one<36>(args, sm_count, st);
    case 40: return launch_one<40>(args, sm_count, st);
    case 44: return launch_one<44>(args, sm_count, st);
    case 48: return launch_one<48>(args, sm_count, st);
    case 52: return launch_one<52>(args, sm_count, st);
    case 56: return launch_one<56>(args, sm_count, st);
    case 60: return launch_one<60>(args, sm_count, st);
    case 64: return launch_one<64>(args, sm_count, st);
    default:
        set_error("adapter too long for the packed DP kernel");
        return VFB_ERR_ARG;
    }
}

uint32_t dp_lcap(const DpLayout &lay, uint32_t A, int extend) { return dp_layout_lcap(lay, A, extend); }

// ---------------------------------------------------------------------------------------
// Fallback: unpacked int32 transcription of the rule set, state in global scratch
// (interleaved across threads).  Any adapter length up to VFB_MAX_ADAPTER, any scores whose
// sums fit int32.  Slow; exists so that no parameter combination leaves the GPU.
#define DPG_THREADS 64
#define DPG_NEG (INT_MIN / 2)

__global__ void __launch_bounds__(DPG_THREADS)
k2_dp_generic(const __grid_constant__ DpGenericJob gj)
{
    const DpJob &job = gj.base;
    const uint32_t n_items = *job.n_items;
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t nth = gj.n_threads;
    const int A = (int)job.adapter_len;
    int32_t *Hs = gj.scratch + (size_t)0 * A * nth + tid;
    int32_t *HLs = gj.scratch + (size_t)1 * A * nth + tid;
    int32_t *Es = gj.scratch + (size_t)2 * A * nth + tid;
    int32_t *ELs = gj.scratch + (size_t)3 * A * nth + tid;
    const int o = gj.sc.open, e = gj.sc.extend;
    for (uint32_t item = tid; item < n_items; item += nth) {
        const uint32_t r = job.worklist[item];
        const vfb_span sp = job.spans[r];
        const int L = (int)sp.len;
        if (L == 0) continue;
        if (job.cells) atomicAdd(job.cells, (unsigned long long)L * (unsigned long long)A);
        for (int i = 0; i < A; ++i) {
            Hs[(size_t)i * nth] = 0; HLs[(size_t)i * nth] = 0;
            Es[(size_t)i * nth] = DPG_NEG; ELs[(size_t)i * nth] = 0;
        }
        int best = DPG_NEG, bestlen = 0, bestj = 0;
        for (int j = 1; j <= L; ++j) {
            const int rc = dp_code(job.text[sp.off + j - 1]);
            int hd = 0, hdl = 0, hup = 0, hupl = 0, F = DPG_NEG, FL = 0;
            for (int i = 0; i < A; ++i) {
                const size_t ix = (size_t)i * nth;
                const int hl = Hs[ix], hll = HLs[ix];
                int E = Es[ix], EL = ELs[ix];
                const int eo = hl - o, ee = E - e;
                if (eo > ee) { E = eo; EL = hll + 1; } else { E = ee; EL = EL + 1; }
                const int fo = hup - o, fe = F - e;
                if (fo > fe) { F = fo; FL = hupl + 1; } else { F = fe; FL = FL + 1; }
                const int ac = gj.d_adapter_code[i];
                const int w = (ac == 4 || rc == 4) ? 0 : (ac == rc ? gj.sc.match : gj.sc.mismatch);
                const int d = hd + w;
                int h, hlen;
                if (d >= E && d >= F) { h = d; hlen = hdl + 1; }
                else if (F >= E) { h = F; hlen = FL; }
                else { h = E; hlen = EL; }
                Es[ix] = E; ELs[ix] = EL; Hs[ix] = h; HLs[ix] = hlen;
                hd = hl; hdl = hll; hup = h; hupl = hlen;
            }
            if (hup > best) { best = hup; bestlen = hupl; bestj = j; }
        }
        int cb = DPG_NEG, cbl = 0;
        for (int i = 0; i < A; ++i) {
            const int h = Hs[(size_t)i * nth];
            if (h > cb) { cb = h; cbl = HLs[(size_t)i * nth]; }
        }
        int score = best, len = bestlen;
        if (cb > best || (cb == best && bestj == L)) { score = cb; len = cbl; }
        if (job.diag_score) { job.diag_score[r] = score; job.diag_len[r] = len; }
        if (score >= job.min_accept) {
            if (job.is_prefix) job.bound[r] = (uint32_t)len;
            else if (len <= L) job.bound[r] = (uint32_t)(L - len);
            if (job.next_list && job.other_bound[r] == VFB_NONE) job.next_list[atomicAdd(job.n_next, 1u)] = r;
        }
    }
}

uint32_t dp_generic_threads(int sm_count) { return (uint32_t)sm_count * 2u * DPG_THREADS; }

int launch_dp_generic(const DpGenericJob &job, int sm_count, cudaStream_t st)
{
    k2_dp_generic<<<sm_count * 2, DPG_THREADS, 0, st>>>(job);
    ++g_launches;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

}  // namespace vfb
