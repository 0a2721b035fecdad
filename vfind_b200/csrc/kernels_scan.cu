// K1 — exact adapter scan, fused with the DP worklist build.
//
// Replaces the two `memmem::find(seq, adapter)` calls per read of
// /root/reference/src/lib.rs:148 (called from :278-286): leftmost byte-exact, case-sensitive
// occurrence of each adapter over the whole read.  Output is the region boundary the exact
// hit implies (:151-152): start = pos + A for the prefix, end = pos for the suffix, VFB_NONE
// when there is no exact hit (the DP kernel may fill it in later).  Reads that still need an
// alignment (`aligner?.align`, :155) are appended to the prefix / suffix worklists here.
//
// Three kernels, chosen by launch_scan():
//  * k1_scan_tile (adapters of 15..64 nt whose sampled 8-byte keys are distinct -- the usual case): the text
//    range of a warp's 32 reads is staged in shared memory by one TMA bulk copy, one lane walks one read and
//    looks up an 8-byte key every 8 (16) bytes in a 512-slot perfect hash; candidates are verified after the
//    walk.  HBM-bound by design: every line of the text is read once.  See the comment above the kernel.
//  * k1_scan_fast (7 <= A <= 64 otherwise: short or repetitive adapters): eight lanes own a read; each lane
//    pulls 16-byte aligned chunks of the text with one LDG.128 and tests only every s-th aligned 32-bit word
//    (s = 4, 2 or 1 words, chosen so that every occurrence of the shorter adapter fully contains a sampled
//    word) -- or 8-byte keys -- in a shared-memory hash of the adapters' k-mers; a hit names the adapter
//    offsets it can sit at, and each candidate start is verified against the adapter pre-shifted to the
//    text's word alignment.
//  * k1_scan_general (any adapter length, including 0 and > 64): one warp per read, byte-wise, ballot.
#include "vfb_internal.cuh"

namespace vfb {

#define SCAN_THREADS 256
#define SCAN_WARPS (SCAN_THREADS / 32)
#define SCAN_MAXC 5             // 16-byte chunks covering an adapter of <= 64 bytes at any alignment
#define SCAN_SLOTS 512          // perfect hash of <= 32 four-mers: one probe, no chain
#define WL_BUF 64               // per-warp worklist staging entries

struct ScanTables {
    // 4-mer hash.  e0 slot = {word, kind | adapter << 8 | offset << 16, next word, next-word mask}:
    // kind 1 = the 4-mer sits at ONE (adapter, offset); the word after it in the text must then
    // match the adapter's next bytes (cuts the 1-in-8 false 4-mer hits before any verification);
    // kind 2 = several (adapter, offset) pairs share the 4-mer: their offsets are bit sets in
    // e1 (prefix in bits 0-15, suffix in bits 16-31) and the next-word mask is 0.
    uint4 e0[SCAN_SLOTS];
    uint32_t e1[SCAN_SLOTS];
    // adapters pre-shifted to every position s inside a 16-byte chunk: bytes and byte masks
    uint4 pat[2][16][SCAN_MAXC];
    uint4 msk[2][16][SCAN_MAXC];
};

struct ScanArgs {
    ScanJob job;
    AdapterBytes prefix, suffix;
    uint32_t mult;      // hash multiplier under which the adapters' sampled 4-mers do not collide
    int multi;          // a sampled 4-mer occurs at more than one (adapter, offset)
};

__host__ __device__ __forceinline__ uint32_t hash4(uint32_t w, uint32_t mult) { return (w * mult) >> 23; }
// 8-byte keys (two consecutive text words)
__host__ __device__ __forceinline__ uint32_t hash8_mult2(uint32_t mult) { return mult * 0x85EBCA6Bu + 2u; }
__host__ __device__ __forceinline__ uint32_t hash8(uint32_t w0, uint32_t w1, uint32_t mult, uint32_t mult2)
{
    return (w0 * mult + w1 * mult2) >> 23;
}

__host__ __device__ __forceinline__ uint32_t load_word_le(const uint8_t *b, int i, int n)
{
    // bytes b[i..i+4) little endian, zero outside [0, n)
    uint32_t w = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int p = i + k;
        if (p >= 0 && p < n) w |= (uint32_t)b[p] << (8 * k);
    }
    return w;
}

__device__ void build_tables(ScanTables *T, const AdapterBytes &pre, const AdapterBytes &suf, int max_k, uint32_t mult,
                             bool next_word, bool key8)
{
    for (int i = threadIdx.x; i < SCAN_SLOTS; i += blockDim.x) {
        T->e0[i] = make_uint4(0, 0, 0, 0);
        T->e1[i] = 0;
    }
    for (int i = threadIdx.x; i < 2 * 16 * SCAN_MAXC * 4; i += blockDim.x) {
        // word m of chunk c of adapter x placed at chunk offset s
        const int m = i & 3, c = (i >> 2) % SCAN_MAXC, s = ((i >> 2) / SCAN_MAXC) & 15, x = (i >> 2) / (SCAN_MAXC * 16);
        const AdapterBytes &ad = x ? suf : pre;
        uint32_t w = 0, k = 0;
        for (int b = 0; b < 4; ++b) {
            const int p = c * 16 + m * 4 + b - s;
            if (p >= 0 && p < (int)ad.len) { w |= (uint32_t)ad.b[p] << (8 * b); k |= 0xFFu << (8 * b); }
        }
        reinterpret_cast<uint32_t *>(&T->pat[x][s][c])[m] = w;
        reinterpret_cast<uint32_t *>(&T->msk[x][s][c])[m] = k;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        // Serial insert (<= 32 entries).  Only offsets k < max_k = 4*stride are needed: the FIRST
        // sampled word an occurrence fully contains sits at adapter offset (-p) mod 4*stride,
        // so every occurrence yields exactly one candidate, in exactly one lane.  The same
        // 4-mer at several offsets ORs into one slot.
        for (int x = 0; x < 2; ++x) {
            const AdapterBytes &ad = x ? suf : pre;
            for (int k = 0; k < max_k && k + (key8 ? 8 : 4) <= (int)ad.len; ++k) {
                const uint32_t w = load_word_le(ad.b, k, (int)ad.len);
                const uint32_t w1 = load_word_le(ad.b, k + 4, (int)ad.len);
                const uint32_t h = key8 ? hash8(w, w1, mult, hash8_mult2(mult)) : hash4(w, mult);      // collision-free by choice of mult (host)
                uint4 e = T->e0[h];
                if (e.y == 0) {
                    e.x = w;
                    e.y = 1u | ((uint32_t)x << 8) | ((uint32_t)k << 16);
                    e.z = e.w = 0;
                    if (key8) {
                        e.z = w1;
                        e.w = 0xFFFFFFFFu;
                    } else if (next_word) {
                        e.z = w1;
                        for (int b = 0; b < 4; ++b)
                            if (k + 4 + b < (int)ad.len) e.w |= 0xFFu << (8 * b);
                    }
                } else {
                    e.y = 2u;
                    if (!key8) e.z = e.w = 0;
                }
                T->e0[h] = e;
                T->e1[h] |= 1u << (k + 16 * x);
            }
        }
    }
    __syncthreads();
    // An empty slot gets a key that does not hash to it: a text key equal to it is looked up in
    // another slot, so the probe needs no "occupied" test — one compare decides.
    for (int i = threadIdx.x; i < SCAN_SLOTS; i += blockDim.x) {
        if (T->e0[i].y != 0) continue;
        uint32_t t = 0;
        while ((key8 ? hash8(t, 0u, mult, hash8_mult2(mult)) : hash4(t, mult)) == (uint32_t)i) ++t;
        T->e0[i] = make_uint4(t, 0u, 0u, 0xFFFFFFFFu);
    }
    __syncthreads();
}

// Per-read geometry shared by a lane group: 16-byte aligned base, bytes of the first chunk
// that precede the read, read length.
struct ReadGeom {
    const uint4 *base16;
    uint32_t lead, len;
};

// Verify a candidate start `rel` of adapter x: 16-byte aligned loads against the adapter
// pre-shifted to the candidate's offset inside its chunk.
__device__ __forceinline__ bool verify_at(const ScanTables *T, uint32_t x, uint32_t rel, uint32_t A, const ReadGeom &rg)
{
    const uint32_t abs0 = rg.lead + rel, s = abs0 & 15u;
    const uint4 *src = rg.base16 + (abs0 >> 4);
    const uint32_t nc = (s + A + 15) >> 4;
    uint32_t diff = 0;
    for (uint32_t k = 0; k < nc; ++k) {
        const uint4 t = __ldg(src + k), pt = T->pat[x][s][k], mk = T->msk[x][s][k];
        diff |= ((t.x ^ pt.x) & mk.x) | ((t.y ^ pt.y) & mk.y) | ((t.z ^ pt.z) & mk.z) | ((t.w ^ pt.w) & mk.w);
    }
    return diff == 0;
}

// A hit on a kind-2 slot: the sampled word at `relq` (bytes after the read start, may be
// negative) equals an adapter 4-mer that sits at several (adapter, offset) pairs.  Expand to
// candidate starts and verify them.
__device__ __forceinline__ void hit_expand(const ScanTables *T, uint32_t slot, int relq, const ReadGeom &rg,
                                           uint32_t AP, uint32_t AS, uint32_t &bestP, uint32_t &bestS)
{
    uint32_t m = T->e1[slot];
    while (m) {
        const int b = __ffs((int)m) - 1;
        m &= m - 1;
        const uint32_t x = (uint32_t)b >> 4;
        const int p = relq - (b & 15);
        const uint32_t A = x ? AS : AP;
        if (p < 0 || p + (int)A > (int)rg.len || (uint32_t)p >= (x ? bestS : bestP)) continue;
        if (verify_at(T, x, (uint32_t)p, A, rg)) {
            if (x) bestS = (uint32_t)p; else bestP = (uint32_t)p;
        }
    }
}

// Out-of-line copy of the verification for the (practically never taken) queue-overflow path.
__device__ __noinline__ uint32_t verify_cold(const ScanTables *T, uint32_t x, uint32_t rel, uint32_t A,
                                             const uint4 *base16, uint32_t lead, uint32_t len)
{
    ReadGeom rg;
    rg.base16 = base16; rg.lead = lead; rg.len = len;
    return verify_at(T, x, rel, A, rg) ? 1u : 0u;
}

// One candidate: adapter x starting at p.
__device__ __forceinline__ void hit_check(const ScanTables *T, uint32_t x, int p, const ReadGeom &rg,
                                          uint32_t AP, uint32_t AS, uint32_t &bestP, uint32_t &bestS)
{
    const uint32_t A = x ? AS : AP;
    if (p < 0 || (uint32_t)p + A > rg.len || (uint32_t)p >= (x ? bestS : bestP)) return;
    if (verify_at(T, x, (uint32_t)p, A, rg)) {
        if (x) bestS = (uint32_t)p; else bestP = (uint32_t)p;
    }
}

// A candidate waits in ONE per-lane slot as ((p + 64) << 1 | adapter) and is verified after the
// trip's probes, all lanes together, so that the divergent verify code runs once per trip
// instead of once per probe.  A second candidate in the same lane and trip (rare: a lane's
// three chunks are 128 bytes apart) sends the waiting one through the out-of-line copy.
struct Hits {
    uint32_t pend;
};

template <bool MULTI, bool KEY8>
__device__ __forceinline__ void probe_word(const ScanTables *T, uint32_t mult, uint32_t mult2, uint32_t w, uint32_t wnext, int relq,
                                           const ReadGeom &rg, uint32_t AP, uint32_t AS, Hits &hq,
                                           uint32_t &bestP, uint32_t &bestS)
{
    const uint32_t h = KEY8 ? hash8(w, wnext, mult, mult2) : hash4(w, mult);
    const uint4 e = T->e0[h];
    const uint32_t diff = KEY8 ? ((e.x ^ w) | (e.z ^ wnext)) : ((e.x ^ w) | ((e.z ^ wnext) & e.w));
    if (diff == 0) {
        if (MULTI && (e.y & 0xFFu) != 1u) { hit_expand(T, h, relq, rg, AP, AS, bestP, bestS); return; }
        if (hq.pend != VFB_NONE) {
            const uint32_t x = hq.pend & 1u, A = x ? AS : AP;
            const int p = (int)(hq.pend >> 1) - 64;
            if (p >= 0 && (uint32_t)p + A <= rg.len && (uint32_t)p < (x ? bestS : bestP) &&
                verify_cold(T, x, (uint32_t)p, A, rg.base16, rg.lead, rg.len)) {
                if (x) bestS = (uint32_t)p; else bestP = (uint32_t)p;
            }
        }
        // (p + 64 < 2^31: reads of 2 GiB and more never reach the probes, see the kernel)
        hq.pend = ((uint32_t)(relq - (int)(e.y >> 16) + 64) << 1) | ((e.y >> 8) & 1u);
    }
}

__device__ __forceinline__ void hits_drain(const ScanTables *T, Hits &hq, const ReadGeom &rg, uint32_t AP,
                                           uint32_t AS, uint32_t &bestP, uint32_t &bestS)
{
    if (__any_sync(0xffffffffu, hq.pend != VFB_NONE)) {
        if (hq.pend != VFB_NONE) {
            hit_check(T, hq.pend & 1u, (int)(hq.pend >> 1) - 64, rg, AP, AS, bestP, bestS);
            hq.pend = VFB_NONE;
        }
    }
}

// KEY8: the table is keyed by 8 text bytes (two words), probed at chunk offset 0 (and 8 when
// STRIDE_WORDS == 2): no false hits to speak of, and duplicates among the adapters' keys are
// rare.  Otherwise 4-byte keys probed every STRIDE_WORDS words, with the next-word check.
template <int STRIDE_WORDS, bool MULTI, bool KEY8>
__device__ __forceinline__ void probe_chunk(const ScanTables *T, uint32_t mult, uint32_t mult2, const uint4 &v, int relq,
                                            const ReadGeom &rg, uint32_t AP, uint32_t AS, Hits &hq,
                                            uint32_t &bestP, uint32_t &bestS)
{
    // (with STRIDE_WORDS == 1 the word after v.w is in the next chunk: the tables carry no
    // next-word check then, the argument is ignored)
    probe_word<MULTI, KEY8>(T, mult, mult2, v.x, v.y, relq, rg, AP, AS, hq, bestP, bestS);
    if (STRIDE_WORDS <= 2) probe_word<MULTI, KEY8>(T, mult, mult2, v.z, v.w, relq + 8, rg, AP, AS, hq, bestP, bestS);
    if (STRIDE_WORDS == 1) {
        probe_word<MULTI, KEY8>(T, mult, mult2, v.y, v.z, relq + 4, rg, AP, AS, hq, bestP, bestS);
        probe_word<MULTI, KEY8>(T, mult, mult2, v.w, 0u, relq + 12, rg, AP, AS, hq, bestP, bestS);
    }
}

// Per-warp staging of worklist appends: one global atomic per WL_BUF/2..WL_BUF entries.
struct WlStage {
    uint32_t buf[2][WL_BUF];
};

__device__ __forceinline__ void wl_flush(uint32_t *stage, uint32_t &cnt, uint32_t *list, uint32_t *counter, int lane)
{
    if (cnt == 0) return;
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(counter, cnt);
    base = __shfl_sync(0xffffffffu, base, 0);
    for (uint32_t i = lane; i < cnt; i += 32) list[base + i] = stage[i];
    __syncwarp();
    cnt = 0;
}

__device__ __forceinline__ void wl_push(uint32_t *stage, uint32_t &cnt, bool want, uint32_t value,
                                        uint32_t *list, uint32_t *counter, int lane)
{
    const unsigned m = __ballot_sync(0xffffffffu, want);
    if (!m) return;
    if (cnt + __popc(m) > WL_BUF) wl_flush(stage, cnt, list, counter, lane);
    if (want) stage[cnt + __popc(m & ((1u << lane) - 1))] = value;
    cnt += __popc(m);
    __syncwarp();
}

__device__ __forceinline__ uint32_t scan_one(const uint8_t *seq, uint32_t L, const uint8_t *ad,
                                            uint32_t A, int lane)
{
    if (A == 0) return 0;              // an empty needle matches at 0 (memchr convention)
    if (A > L) return VFB_NONE;
    const uint32_t last = L - A;
    const uint8_t a0 = ad[0];
    for (uint32_t base = 0; base <= last; base += 32) {
        const uint32_t p = base + lane;
        bool hit = false;
        if (p <= last && __ldg(seq + p) == a0) {
            hit = true;
            for (uint32_t t = 1; t < A; ++t) {
                if (__ldg(seq + p + t) != ad[t]) { hit = false; break; }
            }
        }
        const unsigned m = __ballot_sync(0xffffffffu, hit);
        if (m) return base + (uint32_t)(__ffs((int)m) - 1);
    }
    return VFB_NONE;
}

__device__ __noinline__ uint2 scan_giant(const uint8_t *seq, uint32_t L, const ScanArgs &args, int lane)
{
    return make_uint2(scan_one(seq, L, args.prefix.b, args.prefix.len, lane),
                      scan_one(seq, L, args.suffix.b, args.suffix.len, lane));
}

#define SCAN_GROUP 8                      // lanes per read
#define SCAN_RPW (32 / SCAN_GROUP)        // reads per warp trip

// MULTI = some 4-mer sits at several (adapter, offset) pairs (repetitive or overlapping
// adapters; decided on the host): only then is the kind-2 expansion compiled in.
template <int STRIDE_WORDS, bool MULTI, bool KEY8>
__global__ void __launch_bounds__(SCAN_THREADS, MULTI ? 3 : 4)
k1_scan_fast(const __grid_constant__ ScanArgs args)
{
    __shared__ ScanTables T;
    __shared__ WlStage stage[SCAN_WARPS];
    build_tables(&T, args.prefix, args.suffix, 4 * STRIDE_WORDS, args.mult, STRIDE_WORDS >= 2, KEY8);
    const uint32_t mult = args.mult, mult2 = hash8_mult2(args.mult);
    const ScanJob &job = args.job;
    const uint32_t AP = args.prefix.len, AS = args.suffix.len;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane & (SCAN_GROUP - 1), grp = lane / SCAN_GROUP;
    uint32_t cntP = 0, cntS = 0;
    const uint32_t warps_total = gridDim.x * SCAN_WARPS;
    const uint32_t n_units = (job.n_reads + SCAN_RPW - 1) / SCAN_RPW;
    for (uint32_t unit = blockIdx.x * SCAN_WARPS + warp; unit < n_units; unit += warps_total) {
        const uint32_t r = unit * SCAN_RPW + grp;
        const bool have = r < job.n_reads;
        const vfb_span sp = have ? job.spans[r] : vfb_span{0u, 0u};
        const uintptr_t addr = reinterpret_cast<uintptr_t>(job.text + sp.off);
        ReadGeom rg;
        rg.base16 = reinterpret_cast<const uint4 *>(addr & ~(uintptr_t)15);
        rg.lead = (uint32_t)(addr & 15u);
        rg.len = sp.len;
        uint32_t bestP = VFB_NONE, bestS = VFB_NONE;
        // candidate starts are queued in 31 bits: a read of 2 GiB or more (there can be one in a
        // 4 GiB buffer) is scanned byte-wise by the whole warp instead
        const bool giant = sp.len >= 0x7FFFFF00u;
        if (__any_sync(0xffffffffu, giant)) {
            for (int q = 0; q < SCAN_RPW; ++q) {
                if (!__shfl_sync(0xffffffffu, (int)giant, q * SCAN_GROUP)) continue;
                const uint32_t off = __shfl_sync(0xffffffffu, sp.off, q * SCAN_GROUP);
                const uint32_t ln = __shfl_sync(0xffffffffu, sp.len, q * SCAN_GROUP);
                const uint2 b = scan_giant(job.text + off, ln, args, lane);
                if (grp == q) { bestP = b.x; bestS = b.y; }
            }
        }
        Hits hq{VFB_NONE};
        const uint32_t n_chunks = sp.len && !giant ? (rg.lead + sp.len + 15) >> 4 : 0;
        // warp-uniform trip count: every lane takes part in the converged drain
        const uint32_t max_chunks = __reduce_max_sync(0xffffffffu, n_chunks);
        for (uint32_t cb = 0; cb < max_chunks; cb += 3 * SCAN_GROUP) {
            // three chunks per lane per trip; all loads are issued before any probe
            const uint32_t c0 = cb + g, c1 = c0 + SCAN_GROUP, c2 = c0 + 2 * SCAN_GROUP;
            const uint4 z = make_uint4(0, 0, 0, 0);
            const uint4 v0 = c0 < n_chunks ? __ldg(rg.base16 + c0) : z;
            const uint4 v1 = c1 < n_chunks ? __ldg(rg.base16 + c1) : z;
            const uint4 v2 = c2 < n_chunks ? __ldg(rg.base16 + c2) : z;
            probe_chunk<STRIDE_WORDS, MULTI, KEY8>(&T, mult, mult2, v0, (int)(c0 * 16) - (int)rg.lead, rg, AP, AS, hq, bestP, bestS);
            // (chunks past a read's end were loaded as zeros and cannot pass the bounds check of a hit:
            // the probes need no per-lane guard, only these warp-uniform ones)
            if (cb + SCAN_GROUP < max_chunks)
                probe_chunk<STRIDE_WORDS, MULTI, KEY8>(&T, mult, mult2, v1, (int)(c1 * 16) - (int)rg.lead, rg, AP, AS, hq, bestP, bestS);
            if (cb + 2 * SCAN_GROUP < max_chunks)
                probe_chunk<STRIDE_WORDS, MULTI, KEY8>(&T, mult, mult2, v2, (int)(c2 * 16) - (int)rg.lead, rg, AP, AS, hq, bestP, bestS);
            hits_drain(&T, hq, rg, AP, AS, bestP, bestS);
        }
        // leftmost over the lane group
#pragma unroll
        for (int o = SCAN_GROUP / 2; o > 0; o >>= 1) {
            bestP = min(bestP, __shfl_xor_sync(0xffffffffu, bestP, o));
            bestS = min(bestS, __shfl_xor_sync(0xffffffffu, bestS, o));
        }
        const bool leader = g == 0 && have;
        const uint32_t start = bestP == VFB_NONE ? VFB_NONE : bestP + AP;
        if (leader) {
            job.start[r] = start;
            job.end[r] = bestS;
        }
        // worklists (`aligner?.align` only on an exact miss, src/lib.rs:155)
        const bool needP = leader && job.list_pre && start == VFB_NONE && sp.len > 0;
        const bool needS = leader && job.list_suf && bestS == VFB_NONE && sp.len > 0 &&
                           (job.compute_all || start != VFB_NONE);
        wl_push(stage[warp].buf[0], cntP, needP, r, job.list_pre, job.n_pre, lane);
        wl_push(stage[warp].buf[1], cntS, needS, r, job.list_suf, job.n_suf, lane);
    }
    wl_flush(stage[warp].buf[0], cntP, job.list_pre, job.n_pre, lane);
    wl_flush(stage[warp].buf[1], cntS, job.list_suf, job.n_suf, lane);
}

// ---------------------------------------------------------------------------------------
// Tile kernel (adapters of 15..64 nt whose sampled 8-byte keys are all distinct): the warp's 32
// reads are staged in shared memory by ONE bulk copy (TMA, cp.async.bulk global -> shared,
// completion on an mbarrier) of the contiguous text range that covers them, so HBM is read in
// whole lines exactly once; then one lane owns one read and walks it in 16-byte chunks out of
// shared memory.  Per sampled key: p = w0*m1 + w1*m2, slot p >> 23 of a 512-entry perfect hash
// {p, adapter | offset << 8}; one compare.  A hit is only remembered (the leftmost candidate
// per adapter); the candidates are verified byte-exactly once, after the walk, by all lanes
// together.  A unit whose text range does not fit the tile (wildly scattered spans, giant
// reads) is scanned byte-wise by the whole warp.
#define TILE_WARPS_MAX 8
#define TILE_SLACK 16            // bytes past a tile: the verify's unaligned word reads stay inside the allocation

struct TileTables {
    uint2 slot[SCAN_SLOTS];
    uint32_t adw[2][16];         // adapters as little-endian words, zero padded
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
// the table never changes after the block's set-up: a plain (schedulable) shared load by address
__device__ __forceinline__ uint2 lds64(uint32_t addr)
{
    uint2 r;
    asm("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(r.x), "=r"(r.y) : "r"(addr));
    return r;
}

__device__ __forceinline__ bool tile_verify(const uint32_t *tile32, uint32_t byte_off, const uint32_t *adw, uint32_t A)
{
    const uint32_t sh = (byte_off & 3u) * 8u;
    const uint32_t *p = tile32 + (byte_off >> 2);
    const uint32_t nw = (A + 3) >> 2;
    uint32_t lo = p[0], diff = 0;
    for (uint32_t k = 0; k < nw; ++k) {
        const uint32_t hi = p[k + 1];
        const uint32_t w = __funnelshift_r(lo, hi, sh);
        const uint32_t left = A - 4 * k;
        const uint32_t m = left >= 4 ? 0xFFFFFFFFu : (1u << (8 * left)) - 1u;
        diff |= (w ^ adw[k]) & m;
        lo = hi;
    }
    return diff == 0;
}

// candidate (start + 64) -> verified start or VFB_NONE
__device__ __forceinline__ uint32_t tile_check(const uint32_t *tile32, uint32_t toff, uint32_t len, uint32_t pend,
                                               const uint32_t *adw, uint32_t A)
{
    if (pend == VFB_NONE) return VFB_NONE;
    const int s = (int)pend - 64;
    if (s < 0 || (uint32_t)s + A > len) return VFB_NONE;
    return tile_verify(tile32, toff + (uint32_t)s, adw, A) ? (uint32_t)s : VFB_NONE;
}

// A second candidate for an adapter while one is waiting (a repeated adapter or a false key hit):
// candidates arrive left to right, so the waiting one wins if it verifies.
__device__ __noinline__ uint32_t tile_second(const uint32_t *tile32, uint32_t toff, uint32_t len, uint32_t pend,
                                             uint32_t cand, const uint32_t *adw, uint32_t A)
{
    return tile_check(tile32, toff, len, pend, adw, A) != VFB_NONE ? pend : cand;
}

template <bool STRIDE16>
__global__ void __launch_bounds__(TILE_WARPS_MAX * 32)
k1_scan_tile(const __grid_constant__ ScanArgs args, const uint32_t tile_bytes)
{
    extern __shared__ __align__(128) uint8_t tiles[];
    __shared__ TileTables Ts;
    __shared__ uint32_t stage_all[TILE_WARPS_MAX * 2 * WL_BUF];
    __shared__ unsigned long long bars[TILE_WARPS_MAX];
    TileTables *T = &Ts;
    const int n_warps = blockDim.x >> 5;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t mult = args.mult, mult2 = hash8_mult2(args.mult);
    const uint32_t AP = args.prefix.len, AS = args.suffix.len;

    for (int i = threadIdx.x; i < SCAN_SLOTS; i += blockDim.x)
        T->slot[i] = make_uint2(((uint32_t)i ^ 1u) << 23, 0u);       // a tag that hashes elsewhere: never equal
    for (int i = threadIdx.x; i < 32; i += blockDim.x) {
        const AdapterBytes &ad = (i >> 4) ? args.suffix : args.prefix;
        T->adw[i >> 4][i & 15] = load_word_le(ad.b, 4 * (i & 15), (int)ad.len);
    }
    if (lane == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bars + warp)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const int max_k = STRIDE16 ? 16 : 8;
        for (int x = 0; x < 2; ++x) {
            const AdapterBytes &ad = x ? args.suffix : args.prefix;
            for (int k = 0; k < max_k && k + 8 <= (int)ad.len; ++k) {
                const uint32_t p = load_word_le(ad.b, k, (int)ad.len) * mult + load_word_le(ad.b, k + 4, (int)ad.len) * mult2;
                T->slot[p >> 23] = make_uint2(p, (uint32_t)x | ((uint32_t)k << 8));
            }
        }
    }
    __syncthreads();

    const ScanJob &job = args.job;
    uint32_t *stageP = stage_all + warp * 2 * WL_BUF, *stageS = stageP + WL_BUF;
    uint8_t *tile = tiles + (size_t)warp * (tile_bytes + TILE_SLACK);
    const uint32_t *tile32 = reinterpret_cast<const uint32_t *>(tile);
    const uint32_t bar = smem_u32(bars + warp), tile_s = smem_u32(tile);
    uint32_t slot_s;                                   // kept in a register (opaque: no re-derivation per chunk)
    asm volatile("mov.u32 %0, %1;" : "=r"(slot_s) : "r"(smem_u32(Ts.slot)));
    uint32_t cntP = 0, cntS = 0, parity = 0;
    const uint32_t n_units = (job.n_reads + 31) / 32;
    // the next unit's spans are fetched while the current unit is staged and scanned
    const uint32_t unit_stride = gridDim.x * n_warps;
    vfb_span nsp = vfb_span{0u, 0u};
    {
        const uint32_t r0 = (blockIdx.x * n_warps + warp) * 32 + lane;
        if (r0 < job.n_reads) nsp = job.spans[r0];
    }
    for (uint32_t unit = blockIdx.x * n_warps + warp; unit < n_units; unit += unit_stride) {
        const uint32_t r = unit * 32 + lane;
        const bool have = r < job.n_reads;
        const vfb_span sp = nsp;
        {
            const uint32_t rn = (unit + unit_stride) * 32 + lane;
            nsp = vfb_span{0u, 0u};
            if (unit + unit_stride < n_units && rn < job.n_reads) nsp = job.spans[rn];
        }
        const bool live = have && sp.len > 0;
        const uint32_t lo = __reduce_min_sync(0xffffffffu, live ? sp.off : 0xFFFFFFFFu);
        const uint32_t last = __reduce_max_sync(0xffffffffu, live ? sp.off + (sp.len - 1) : 0u);
        uint32_t bestP = VFB_NONE, bestS = VFB_NONE;
        if (lo != 0xFFFFFFFFu) {
            const uintptr_t g0 = reinterpret_cast<uintptr_t>(job.text + lo);
            const uint32_t lead_tile = (uint32_t)(g0 & 15u);
            const uint64_t n_bytes = ((uint64_t)(last - lo) + 1 + lead_tile + 15) & ~15ull;
            if (n_bytes <= tile_bytes) {
                __syncwarp();                      // every lane is done with the previous unit's tile
                if (lane == 0) {
                    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)n_bytes) : "memory");
                    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                 ::"r"(tile_s), "l"(g0 & ~(uintptr_t)15), "r"((uint32_t)n_bytes), "r"(bar) : "memory");
                }
                uint32_t ok;
                do {
                    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
                } while (!ok);
                parity ^= 1u;
                if (live) {
                    const uint32_t toff = lead_tile + (sp.off - lo);       // the read inside the tile
                    const uint32_t lead = toff & 15u;
                    const uint4 *tp = reinterpret_cast<const uint4 *>(tile) + (toff >> 4);
                    const uint32_t nch = (lead + sp.len + 15) >> 4;
                    uint32_t pendP = VFB_NONE, pendS = VFB_NONE;
                    int relq = 64 - (int)lead;                             // candidate starts are kept + 64
                    auto hit = [&](uint32_t meta, int at) {
                        const uint32_t cand = (uint32_t)(at - (int)(meta >> 8));
                        if (meta & 1u)
                            pendS = pendS == VFB_NONE ? cand : tile_second(tile32, toff, sp.len, pendS, cand, Ts.adw[1], AS);
                        else
                            pendP = pendP == VFB_NONE ? cand : tile_second(tile32, toff, sp.len, pendP, cand, Ts.adw[0], AP);
                    };
#pragma unroll 2
                    for (uint32_t c = 0; c < nch; ++c, relq += 16) {
                        const uint4 v = tp[c];
                        const uint32_t p0 = v.x * mult + v.y * mult2;
                        const uint2 e0 = lds64(slot_s + ((p0 >> 23) << 3));
                        if (STRIDE16) {
                            if (e0.x == p0) hit(e0.y, relq);
                        } else {
                            const uint32_t p1 = v.z * mult + v.w * mult2;
                            const uint2 e1 = lds64(slot_s + ((p1 >> 23) << 3));
                            if (e0.x == p0 || e1.x == p1) {                // one (rarely taken) branch per chunk
                                if (e0.x == p0) hit(e0.y, relq);
                                if (e1.x == p1) hit(e1.y, relq + 8);
                            }
                        }
                    }
                    bestP = tile_check(tile32, toff, sp.len, pendP, T->adw[0], AP);
                    bestS = tile_check(tile32, toff, sp.len, pendS, T->adw[1], AS);
                }
            } else {
                // the unit's reads are too far apart for a tile: byte-wise, the whole warp per read
                unsigned todo = __ballot_sync(0xffffffffu, live);
                while (todo) {
                    const int q = __ffs((int)todo) - 1;
                    todo &= todo - 1;
                    const uint32_t off = __shfl_sync(0xffffffffu, sp.off, q);
                    const uint32_t ln = __shfl_sync(0xffffffffu, sp.len, q);
                    const uint2 b = scan_giant(job.text + off, ln, args, lane);
                    if (lane == q) { bestP = b.x; bestS = b.y; }
                }
            }
        }
        const uint32_t start = bestP == VFB_NONE ? VFB_NONE : bestP + AP;
        if (have) {
            job.start[r] = start;
            job.end[r] = bestS;
        }
        const bool needP = live && job.list_pre && start == VFB_NONE;
        const bool needS = live && job.list_suf && bestS == VFB_NONE && (job.compute_all || start != VFB_NONE);
        wl_push(stageP, cntP, needP, r, job.list_pre, job.n_pre, lane);
        wl_push(stageS, cntS, needS, r, job.list_suf, job.n_suf, lane);
    }
    wl_flush(stageP, cntP, job.list_pre, job.n_pre, lane);
    wl_flush(stageS, cntS, job.list_suf, job.n_suf, lane);
}

// Tile size for a batch whose reads sit `stride` bytes apart on average: 32 reads and a little slack.
uint32_t vfb_tile_bytes_for(uint64_t text_bytes, uint32_t n_reads)
{
    uint64_t stride = n_reads ? text_bytes / n_reads : 0;
    if (stride < 32) stride = 32;
    uint64_t t = 32 * stride + stride + 64;
    t = (t + 127) & ~127ull;
    if (t < 2048) t = 2048;
    if (t > VFB_TILE_BYTES_MAX) t = VFB_TILE_BYTES_MAX;
    return (uint32_t)t;
}

// Shared memory of a tile block of `w` warps: their tiles (dynamic), the tables, worklist stages and barriers, and a
// reserve.
static constexpr size_t scan_tile_block_smem(size_t tile, int w)
{
    return (size_t)w * (tile + TILE_SLACK) + sizeof(TileTables) + TILE_WARPS_MAX * (2 * WL_BUF * 4 + 8) + 1024;
}
static_assert(scan_tile_block_smem(VFB_TILE_BYTES_MAX, 1) <= VFB_SMEM_BLOCK_MAX, "a block of one warp fits any tile");

template <bool STRIDE16>
static int launch_scan_tile(const ScanArgs &a, int sm_count, cudaStream_t st)
{
    const uint32_t tile = vfb_tile_bytes_for(a.job.text_bytes, a.job.n_reads);
    // as many warps per SM as the tiles allow, in blocks of 8 / 4 / 2 / 1 warps
    int warps = 1, best_total = 0;
    for (int w = TILE_WARPS_MAX; w >= 1; w >>= 1) {
        int bps = (int)(VFB_SMEM_BLOCK_MAX / scan_tile_block_smem(tile, w));
        if (bps * w > 32) bps = 32 / w;            // 1024 resident threads are plenty
        if (bps * w > best_total) { best_total = bps * w; warps = w; }
    }
    const size_t smem = (size_t)warps * (tile + TILE_SLACK);
    const int bps = best_total / warps;
    VFB_CUDA(cudaFuncSetAttribute(k1_scan_tile<STRIDE16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const uint32_t units = (a.job.n_reads + 31) / 32;
    uint32_t blocks = (units + warps - 1) / warps;
    const uint32_t cap = (uint32_t)sm_count * (uint32_t)bps;
    if (blocks > cap) blocks = cap;
    k1_scan_tile<STRIDE16><<<blocks, warps * 32, smem, st>>>(a, tile);
    return VFB_OK;
}

// ---------------------------------------------------------------------------------------
// General kernel: any adapter length (including 0 and > 64).  One warp per read; lanes test
// consecutive start positions byte by byte and vote.
__global__ void __launch_bounds__(SCAN_THREADS)
k1_scan_general(const __grid_constant__ ScanArgs args)
{
    __shared__ uint8_t s_pre[VFB_MAX_SCAN_ADAPTER], s_suf[VFB_MAX_SCAN_ADAPTER];
    __shared__ WlStage stage[SCAN_WARPS];
    for (uint32_t i = threadIdx.x; i < args.prefix.len; i += blockDim.x) s_pre[i] = args.prefix.b[i];
    for (uint32_t i = threadIdx.x; i < args.suffix.len; i += blockDim.x) s_suf[i] = args.suffix.b[i];
    __syncthreads();
    const ScanJob &job = args.job;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t cntP = 0, cntS = 0;
    const uint32_t warps_total = gridDim.x * SCAN_WARPS;
    for (uint32_t r = blockIdx.x * SCAN_WARPS + warp; r < job.n_reads; r += warps_total) {
        const vfb_span sp = job.spans[r];
        const uint8_t *seq = job.text + sp.off;
        const uint32_t pp = scan_one(seq, sp.len, s_pre, args.prefix.len, lane);
        const uint32_t ps = scan_one(seq, sp.len, s_suf, args.suffix.len, lane);
        const uint32_t start = pp == VFB_NONE ? VFB_NONE : pp + args.prefix.len;
        if (lane == 0) {
            job.start[r] = start;
            job.end[r] = ps;
        }
        const bool needP = lane == 0 && job.list_pre && start == VFB_NONE && sp.len > 0;
        const bool needS = lane == 0 && job.list_suf && ps == VFB_NONE && sp.len > 0 &&
                           (job.compute_all || start != VFB_NONE);
        wl_push(stage[warp].buf[0], cntP, needP, r, job.list_pre, job.n_pre, lane);
        wl_push(stage[warp].buf[1], cntS, needS, r, job.list_suf, job.n_suf, lane);
    }
    wl_flush(stage[warp].buf[0], cntP, job.list_pre, job.n_pre, lane);
    wl_flush(stage[warp].buf[1], cntS, job.list_suf, job.n_suf, lane);
}

int launch_scan(const ScanJob &job, const AdapterBytes &prefix, const AdapterBytes &suffix,
                int sm_count, cudaStream_t st)
{
    if (job.n_reads == 0) return VFB_OK;
    ScanArgs a;
    a.job = job;
    a.prefix = prefix;
    a.suffix = suffix;
    const uint32_t amin = prefix.len < suffix.len ? prefix.len : suffix.len;
    const uint32_t amax = prefix.len > suffix.len ? prefix.len : suffix.len;
    bool fast = amin >= 7 && amax <= 64 && !job.force_general;
    bool key8 = false;
    int stride_words = 1;
    if (fast) {
        // perfect hash: find a multiplier under which the sampled 4-mers of both adapters
        // occupy distinct slots (<= 32 keys in 512 slots: a few tries)
        // amin >= 23: 8-byte keys every 16 bytes; >= 15: 8-byte keys every 8 bytes; >= 11: 4-byte keys
        // every 8 bytes; else 4-byte keys every 4 bytes (every occurrence of the shorter adapter
        // fully contains a sampled key)
        key8 = amin >= 15;
        stride_words = amin >= 23 ? 4 : (amin >= 11 ? 2 : 1);
        const int max_k = 4 * stride_words, klen = key8 ? 8 : 4;
        bool ok = false;
        bool multi = false;
        for (uint32_t t = 0; t < 4096 && !ok; ++t) {
            const uint32_t mult = 0x9E3779B1u + 2u * t * 0x632BE5ABu;
            uint32_t w0s[SCAN_SLOTS], w1s[SCAN_SLOTS];
            bool used[SCAN_SLOTS] = {false};
            ok = true;
            multi = false;
            for (int x = 0; x < 2 && ok; ++x) {
                const AdapterBytes &ad = x ? suffix : prefix;
                for (int k = 0; k < max_k && k + klen <= (int)ad.len; ++k) {
                    const uint32_t w = load_word_le(ad.b, k, (int)ad.len);
                    const uint32_t w1 = key8 ? load_word_le(ad.b, k + 4, (int)ad.len) : 0u;
                    const uint32_t h = key8 ? hash8(w, w1, mult, hash8_mult2(mult)) : hash4(w, mult);
                    if (used[h] && (w0s[h] != w || w1s[h] != w1)) { ok = false; break; }
                    if (used[h]) multi = true;
                    used[h] = true;
                    w0s[h] = w;
                    w1s[h] = w1;
                }
            }
            if (ok) a.mult = mult;
        }
        fast = ok;
        a.multi = multi ? 1 : 0;
    }
    const uint32_t units = fast ? (job.n_reads + SCAN_RPW - 1) / SCAN_RPW : job.n_reads;
    uint32_t blocks = (units + SCAN_WARPS - 1) / SCAN_WARPS;
    const uint32_t cap = (uint32_t)sm_count * 8u;
    if (blocks > cap) blocks = cap;
#define VFB_SCAN_LAUNCH(S)                                                                  \
    do {                                                                                    \
        if (a.multi) k1_scan_fast<S, true, false><<<blocks, SCAN_THREADS, 0, st>>>(a);      \
        else k1_scan_fast<S, false, false><<<blocks, SCAN_THREADS, 0, st>>>(a);             \
    } while (0)
    if (!fast) k1_scan_general<<<blocks, SCAN_THREADS, 0, st>>>(a);
    else if (key8 && !a.multi) {
        const int rc = stride_words == 4 ? launch_scan_tile<true>(a, sm_count, st) : launch_scan_tile<false>(a, sm_count, st);
        if (rc) return rc;
    } else if (key8 && stride_words == 4) k1_scan_fast<4, true, true><<<blocks, SCAN_THREADS, 0, st>>>(a);
    else if (key8) k1_scan_fast<2, true, true><<<blocks, SCAN_THREADS, 0, st>>>(a);
    else if (stride_words == 2) VFB_SCAN_LAUNCH(2);
    else VFB_SCAN_LAUNCH(1);
#undef VFB_SCAN_LAUNCH
    ++g_launches;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

}  // namespace vfb
