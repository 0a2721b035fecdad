// K3 — variable-region extraction + codon translation + key hashing, and
// K4 — exact on-device counting in an open-addressing table, plus the table utilities the
// multi-GPU merge needs.
//
// K3 replaces the slice of /root/reference/src/lib.rs:288-290 and `translate` (:16-44 with
// the tables at :52-95); K4 replaces `*variants.entry(k).or_insert(0) += 1` (:296, :301) on
// HashMap<String,u64> (:263) and the unzip to columns (:312).
#include "hash.h"
#include "translate_fast.h"
#include "vfb_internal.cuh"

namespace vfb {

// ------------------------------------------------------------------------------------ K3
// AA_TABLE_CANONICAL (src/lib.rs:52-77) flattened as c1*16 + c2*4 + c3, A=0 C=1 G=2 T/U=3.
__constant__ char c_aa[65] =
    "KNKN" "TTTT" "RSRS" "IIMI"
    "QHQH" "PPPP" "RRRR" "LLLL"
    "EDED" "AAAA" "GGGG" "VVVV"
    "*Y*Y" "SSSS" "*CWC" "LFLF";

// ASCII_TO_INDEX (src/lib.rs:86-95); bytes >= 128 are handled before the lookup (:24-29).
__device__ __forceinline__ uint32_t tr_index(uint8_t b)
{
    switch (b) {
    case 'A': case 'a': return 0;
    case 'C': case 'c': return 1;
    case 'G': case 'g': return 2;
    case 'T': case 't': case 'U': case 'u': return 3;
    default: return 4;
    }
}

// String::from_utf8 validity (src/lib.rs:295), sequential; only runs when a region holds
// a byte >= 0x80.
__device__ bool utf8_valid(const uint8_t *s, uint32_t n)
{
    uint32_t i = 0;
    while (i < n) {
        const uint8_t b = s[i];
        if (b < 0x80) { ++i; continue; }
        if (b >= 0xC2 && b <= 0xDF) {
            if (i + 1 >= n || (s[i + 1] & 0xC0) != 0x80) return false;
            i += 2;
        } else if (b >= 0xE0 && b <= 0xEF) {
            if (i + 2 >= n) return false;
            const uint8_t b1 = s[i + 1], b2 = s[i + 2];
            if ((b1 & 0xC0) != 0x80 || (b2 & 0xC0) != 0x80) return false;
            if (b == 0xE0 && b1 < 0xA0) return false;
            if (b == 0xED && b1 > 0x9F) return false;
            i += 3;
        } else if (b >= 0xF0 && b <= 0xF4) {
            if (i + 3 >= n) return false;
            const uint8_t b1 = s[i + 1], b2 = s[i + 2], b3 = s[i + 3];
            if ((b1 & 0xC0) != 0x80 || (b2 & 0xC0) != 0x80 || (b3 & 0xC0) != 0x80) return false;
            if (b == 0xF0 && b1 < 0x90) return false;
            if (b == 0xF4 && b1 > 0x8F) return false;
            i += 4;
        } else {
            return false;
        }
    }
    return true;
}

#define KEY_MULTS 128               // hash multipliers kept in shared memory

// ---- k3_keys_tile: the text range that covers the regions of a warp's 32 reads is staged in shared
// memory by one bulk copy (TMA, completion on an mbarrier), as in k1_scan_tile; one lane owns one read
// and walks its region out of shared memory (no global-load latency inside the translate loop); the
// unit's keys are assembled in shared memory and leave with coalesced 16-byte stores; koff / klen /
// khash are written one lane per read.  A unit whose regions do not fit the tile reads global memory
// directly, a unit whose keys do not fit the key staging writes them directly.
#define K3T_WARPS_MAX 8
#define K3T_OUT_BYTES 4096
#define K3T_SLACK 16

struct Key3Tables {
    uint8_t lut25[256], lut5[256], lut1[256];
    uint8_t aa[128];
    uint64_t mult[KEY_MULTS];
};

__device__ __forceinline__ uint32_t k3_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// aligned word `idx` of the region's source: shared-memory tile, or global memory never touching a word
// at or beyond `limit`
template <bool SMEM>
__device__ __forceinline__ uint32_t k3_word(const uint32_t *w, uint32_t idx, const uint32_t *limit)
{
    if (SMEM) return w[idx];
    return (w + idx) < limit ? __ldg(w + idx) : 0u;
}

// One lane translates (or copies) its region into key words; returns the hash accumulator.
template <bool SMEM, bool TRANSLATE>
__device__ __forceinline__ uint64_t k3_lane(const Key3Tables &T, const uint32_t *w, const uint32_t *limit, uint32_t sh,
                                            uint32_t kl, uint32_t *out, uint32_t &high)
{
    const uint32_t nw = (kl + 3) >> 2, npad = ((kl + 15u) & ~15u) >> 2;
    uint64_t acc = 0;
    uint32_t t0 = k3_word<SMEM>(w, 0, limit), wp = 1;
    for (uint32_t wi = 0; wi < nw; ++wi) {
        uint32_t word;
        if (TRANSLATE) {
            const uint32_t t1 = k3_word<SMEM>(w, wp, limit), t2 = k3_word<SMEM>(w, wp + 1, limit), t3 = k3_word<SMEM>(w, wp + 2, limit);
            wp += 3;
            const uint32_t x0 = __funnelshift_r(t0, t1, sh), x1 = __funnelshift_r(t1, t2, sh), x2 = __funnelshift_r(t2, t3, sh);
            t0 = t3;
            // codon a = bytes 3a .. 3a+2 of the 12 (translate, src/lib.rs:16-44)
            const uint32_t i0 = T.lut25[x0 & 0xFFu] + T.lut5[(x0 >> 8) & 0xFFu] + T.lut1[(x0 >> 16) & 0xFFu];
            const uint32_t i1 = T.lut25[x0 >> 24] + T.lut5[x1 & 0xFFu] + T.lut1[(x1 >> 8) & 0xFFu];
            const uint32_t i2 = T.lut25[(x1 >> 16) & 0xFFu] + T.lut5[x1 >> 24] + T.lut1[x2 & 0xFFu];
            const uint32_t i3 = T.lut25[(x2 >> 8) & 0xFFu] + T.lut5[(x2 >> 16) & 0xFFu] + T.lut1[x2 >> 24];
            word = (uint32_t)T.aa[i0] | ((uint32_t)T.aa[i1] << 8) | ((uint32_t)T.aa[i2] << 16) | ((uint32_t)T.aa[i3] << 24);
        } else {
            const uint32_t t1 = k3_word<SMEM>(w, wp, limit);
            wp += 1;
            word = __funnelshift_r(t0, t1, sh);
            t0 = t1;
        }
        const uint32_t left = kl - 4 * wi;                 // key bytes from this word on, >= 1
        if (left < 4) word &= (1u << (8 * left)) - 1u;
        if (!TRANSLATE) high |= word & 0x80808080u;
        acc += (uint64_t)(word ^ VFB_HASH_K) * (wi < KEY_MULTS ? T.mult[wi] : vfb_hash_mult(wi));
        out[wi] = word;
    }
    for (uint32_t wi = nw; wi < npad; ++wi) out[wi] = 0u;
    return acc;
}

// umi_length: appends the UMI (ulen bytes at `u`, read from global memory) to a key of kr bytes in out[]: key byte
// kr + j = UMI byte j.  The hash accumulator is updated word by word (the region's partial last word is replaced), and
// the composite key is zero-padded to 16 bytes.  No translation past kr.
__device__ __forceinline__ void umi_append(const uint8_t *u, uint32_t ulen, uint32_t kr, uint32_t *out, uint64_t &acc,
                                           const uint64_t *mult)
{
    const uintptr_t va = reinterpret_cast<uintptr_t>(u);
    const uint32_t *g = reinterpret_cast<const uint32_t *>(va & ~(uintptr_t)3);
    const uint32_t *limit = reinterpret_cast<const uint32_t *>((va + ulen + 3) & ~(uintptr_t)3);
    const uint32_t sh = (uint32_t)(va & 3u) * 8u;
    const uint32_t w0 = kr >> 2, d = kr & 3u, nw = (kr + ulen + 3) >> 2, npad = ((kr + ulen + 15u) & ~15u) >> 2;
    uint32_t prev = 0, g0 = k3_word<false>(g, 0, limit);
    for (uint32_t m = 0; w0 + m < nw; ++m) {
        uint32_t um = 0;                                   // UMI bytes 4m .. 4m+3
        if (4 * m < ulen) {
            const uint32_t g1 = k3_word<false>(g, m + 1, limit);
            um = __funnelshift_r(g0, g1, sh);
            g0 = g1;
            const uint32_t left = ulen - 4 * m;
            if (left < 4) um &= (1u << (8 * left)) - 1u;
        }
        const uint32_t wi = w0 + m;
        uint32_t word = __funnelshift_rc(prev, um, 32u - 8u * d);   // UMI bytes 4m - d .. 4m - d + 3
        const uint64_t M = wi < KEY_MULTS ? mult[wi] : vfb_hash_mult(wi);
        if (m == 0 && d) {
            const uint32_t was = out[wi];
            word |= was;
            acc -= (uint64_t)(was ^ VFB_HASH_K) * M;
        }
        acc += (uint64_t)(word ^ VFB_HASH_K) * M;
        out[wi] = word;
        prev = um;
    }
    for (uint32_t wi = nw; wi < npad; ++wi) out[wi] = 0u;
}

// A read with a key (klen != 0, region at roff, V bytes) gets its UMI appended: klen grows by umi.len and uoff is where
// the UMI sits in the text.  A read shorter than offset + len gets no key and is counted in n_short, unless its region
// is not UTF-8 (a byte key that would not have been counted anyway; only the region is checked).
template <bool TRANSLATE>
__device__ __forceinline__ void umi_plan(const UmiArgs &umi, const KeyJob &job, const vfb_span &sp, uint32_t roff, uint32_t V,
                                         uint32_t &klen, uint32_t &uoff, uint32_t &n_short)
{
    if (!klen) return;
    if (sp.len < umi.offset + umi.len) {
        n_short += (TRANSLATE || utf8_valid(job.text + roff, V)) ? 1u : 0u;
        klen = 0;
    } else {
        klen += umi.len;
        uoff = sp.off + umi.offset;
    }
}

template <bool TRANSLATE, bool UMI>
__global__ void __launch_bounds__(K3T_WARPS_MAX * 32)
k3_keys_tile(const __grid_constant__ KeyJob job, const uint32_t tile_bytes, const __grid_constant__ UmiArgs umi)
{
    extern __shared__ __align__(128) uint8_t dyn[];
    __shared__ Key3Tables T;
    __shared__ unsigned long long bars[K3T_WARPS_MAX];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        const uint32_t c = i >= 128 ? 4u : tr_index((uint8_t)i);
        T.lut25[i] = (uint8_t)(25u * c); T.lut5[i] = (uint8_t)(5u * c); T.lut1[i] = (uint8_t)c;
    }
    for (int i = threadIdx.x; i < 128; i += blockDim.x) {
        const int c0 = i / 25, c1 = (i / 5) % 5, c2 = i % 5;
        T.aa[i] = (i >= 125 || c0 == 4 || c1 == 4 || c2 == 4) ? (uint8_t)'X' : (uint8_t)c_aa[c0 * 16 + c1 * 4 + c2];
    }
    for (int i = threadIdx.x; i < KEY_MULTS; i += blockDim.x) T.mult[i] = vfb_hash_mult((uint32_t)i);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    if (lane == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(k3_smem_u32(bars + warp)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const size_t per_warp = (size_t)tile_bytes + K3T_SLACK + K3T_OUT_BYTES;
    uint8_t *tile = dyn + (size_t)warp * per_warp;
    const uint32_t *tile32 = reinterpret_cast<const uint32_t *>(tile);
    uint32_t *out32 = reinterpret_cast<uint32_t *>(tile + tile_bytes + K3T_SLACK);
    const uint32_t bar = k3_smem_u32(bars + warp), tile_s = k3_smem_u32(tile);
    uint32_t parity = 0;
    uint32_t n_short = 0;                                  // UMI: reads of this warp's units whose UMI does not fit
    const uint32_t n_units = (job.n_reads + 31) / 32;
    for (uint32_t unit = blockIdx.x * n_warps + warp; unit < n_units; unit += gridDim.x * n_warps) {
        // ---- one lane per read: key length, key space (one atomic per 32 reads)
        const uint32_t r = unit * 32 + lane;
        uint32_t klen = 0, V = 0, roff = 0;            // roff: byte offset of the region in the text
        if (r < job.n_reads) {
            const uint32_t s = job.start[r], e = job.end[r];
            // src/lib.rs:288: both located and start < end (strict)
            if (s != VFB_NONE && e != VFB_NONE && s < e) {
                const vfb_span sp = job.spans[r];
                if (e <= sp.len) {
                    V = e - s;
                    roff = sp.off + s;
                    if (!TRANSLATE) klen = V;
                    else if (V % 3 == 0) klen = V / 3;                 // :17-19 partial codon -> None
                }
            }
        }
        uint32_t uoff = 0;                             // UMI: byte offset of the UMI in the text
        if constexpr (UMI) umi_plan<TRANSLATE>(umi, job, job.spans[r], roff, V, klen, uoff, n_short);
        const unsigned owners = __ballot_sync(0xffffffffu, klen != 0);
        if (owners == 0) {
            if (r < job.n_reads) job.klen[r] = 0;
            continue;
        }
        const uint32_t padded = (klen + 15u) & ~15u;
        uint32_t incl = padded;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        unsigned long long base = 0;
        const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
        if (lane == 31) base = atomicAdd(job.key_cursor, (unsigned long long)total);
        base = __shfl_sync(0xffffffffu, base, 31);
        const uint32_t local = incl - padded;              // this lane's key inside the unit's key block
        // ---- stage the text that covers the owners' regions
        const uint32_t lo = __reduce_min_sync(0xffffffffu, klen ? roff : 0xFFFFFFFFu);
        const uint32_t last = __reduce_max_sync(0xffffffffu, klen ? roff + (V - 1) : 0u);
        const uintptr_t g0 = reinterpret_cast<uintptr_t>(job.text + lo);
        const uint32_t lead_tile = (uint32_t)(g0 & 15u);
        const uint64_t n_bytes = ((uint64_t)(last - lo) + 1 + lead_tile + 15) & ~15ull;
        const bool staged = n_bytes <= tile_bytes;
        const bool out_staged = total <= K3T_OUT_BYTES;
        __syncwarp();                                      // the previous unit's tile and key block are done with
        if (staged) {
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
        }
        uint64_t acc = 0;
        uint32_t high = 0;
        if (klen) {
            uint32_t *out = out_staged ? out32 + (local >> 2) : reinterpret_cast<uint32_t *>(job.keys + base + local);
            const uint32_t kr = UMI ? klen - umi.len : klen;          // the region's part of the key
            if (staged) {
                const uint32_t toff = lead_tile + (roff - lo);
                acc = k3_lane<true, TRANSLATE>(T, tile32 + (toff >> 2), nullptr, (toff & 3u) * 8u, kr, out, high);
            } else {
                const uintptr_t va = reinterpret_cast<uintptr_t>(job.text + roff);
                const uint32_t *limit = reinterpret_cast<const uint32_t *>((va + V + 3) & ~(uintptr_t)3);
                acc = k3_lane<false, TRANSLATE>(T, reinterpret_cast<const uint32_t *>(va & ~(uintptr_t)3), limit,
                                                (uint32_t)(va & 3u) * 8u, kr, out, high);
            }
            if constexpr (UMI) umi_append(job.text + uoff, umi.len, kr, out, acc, T.mult);
        }
        __syncwarp();
        if (out_staged) {
            const uint4 *src = reinterpret_cast<const uint4 *>(out32);
            uint4 *dst = reinterpret_cast<uint4 *>(job.keys + base);
            for (uint32_t c = lane; c < total / 16; c += 32) dst[c] = src[c];
        }
        if (klen) {
            job.koff[r] = base + local;
            uint64_t h = vfb_hash_finish(acc, klen);
            if (job.hash_bits > 0 && job.hash_bits < 64) h &= (1ull << job.hash_bits) - 1;
            job.khash[r] = h;
            // String::from_utf8 (:295): only regions holding a byte >= 0x80 need the validator
            if (!TRANSLATE && high && !utf8_valid(job.text + roff, V)) klen = 0;
        }
        if (r < job.n_reads) job.klen[r] = klen;
    }
    if constexpr (UMI) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) n_short += __shfl_xor_sync(0xffffffffu, n_short, o);
        if (lane == 0 && n_short) atomicAdd(umi.n_short, (unsigned long long)n_short);
    }
}

// Shared memory of a k3_keys_tile block of `w` warps: their tiles and key staging (dynamic), the tables and barriers,
// and a reserve.
static constexpr size_t keys_tile_block_smem(size_t tile, int w)
{
    return (size_t)w * (tile + K3T_SLACK + K3T_OUT_BYTES) + sizeof(Key3Tables) + 64 + 1024;
}
static_assert(keys_tile_block_smem(VFB_TILE_BYTES_MAX, 1) <= VFB_SMEM_BLOCK_MAX, "a block of one warp fits any tile");

template <bool TRANSLATE, bool UMI>
static int launch_keys_tile(const KeyJob &job, cudaStream_t st, const UmiArgs &umi)
{
    const uint32_t tile = vfb_tile_bytes_for(job.text_bytes, job.n_reads);
    int best_w = 1, best_total = 0;
    for (int w = K3T_WARPS_MAX; w >= 1; w >>= 1) {
        int bps = (int)(VFB_SMEM_BLOCK_MAX / keys_tile_block_smem(tile, w));
        if (bps * w > 32) bps = 32 / w;
        if (bps * w > best_total) { best_total = bps * w; best_w = w; }
    }
    const size_t smem = (size_t)best_w * (tile + K3T_SLACK + K3T_OUT_BYTES);
    VFB_CUDA(cudaFuncSetAttribute(k3_keys_tile<TRANSLATE, UMI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const uint32_t units = (job.n_reads + 31) / 32;
    uint32_t blocks = (units + best_w - 1) / best_w;
    const uint32_t cap = 148u * (uint32_t)(best_total / best_w);
    if (blocks > cap) blocks = cap;
    k3_keys_tile<TRANSLATE, UMI><<<blocks, best_w * 32, smem, st>>>(job, tile, umi);
    return VFB_OK;
}

int launch_keys(const KeyJob &job, cudaStream_t st, const UmiArgs &umi)
{
    if (job.n_reads == 0) return VFB_OK;
    int rc;
    if (!umi.len) rc = job.skip_translation ? launch_keys_tile<false, false>(job, st, umi) : launch_keys_tile<true, false>(job, st, umi);
    else rc = job.skip_translation ? launch_keys_tile<false, true>(job, st, umi) : launch_keys_tile<true, true>(job, st, umi);
    if (rc != VFB_OK) return rc;
    ++g_launches;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

// ------------------------------------------------------------------------------------ K4
#define REF_BATCH 0x80000000u

struct InsertArgs {
    DevTable t;
    InsertJob job;
};

__device__ __forceinline__ const uint8_t *job_key(const InsertJob &j, uint32_t i)
{
    return j.koff ? j.keys + j.koff[i] : j.keys + (size_t)i * j.key_stride;
}

// No early exit: a tag match is almost always a key match, so all chunks are needed anyway, and
// without the exit the loads of both keys are in flight together (one memory round trip, not n).
__device__ __forceinline__ bool keys_equal16(const uint8_t *a, const uint8_t *b, uint32_t len)
{
    const uint4 *x = reinterpret_cast<const uint4 *>(a), *y = reinterpret_cast<const uint4 *>(b);
    const uint32_t n = (len + 15) / 16;
    uint32_t diff = 0;
    uint32_t i = 0;
    for (; i + 4 <= n; i += 4) {
        uint4 u[4], v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { u[k] = x[i + k]; v[k] = y[i + k]; }
#pragma unroll
        for (int k = 0; k < 4; ++k)
            diff |= (u[k].x ^ v[k].x) | (u[k].y ^ v[k].y) | (u[k].z ^ v[k].z) | (u[k].w ^ v[k].w);
    }
    for (; i < n; ++i) {
        const uint4 u = x[i], v = y[i];
        diff |= (u.x ^ v.x) | (u.y ^ v.y) | (u.z ^ v.z) | (u.w ^ v.w);
    }
    return diff == 0;
}

// ------------------------------------------------------------------------------------ K3+K4 fused
// k34_keys_count: the key kernel probes the table itself.  A read whose key already has a row (most reads of a
// steady-state batch) is counted right here — its key never leaves shared memory — and only the keys the table
// does not know yet (or whose probe chain is long) are written to the batch's key space and appended to a compact
// list {koff, klen, khash} that k4_insert / k4_publish then work through.  The kernel only READS slots that were
// published by earlier launches (the host orders it behind the previous batch's k4_publish), so a slot is either
// empty or refers to a complete row; counts are added with the same atomics k4_insert uses.
//
// The translate loop takes the arithmetic path of translate_fast.h for twelve canonical bases at a time (one
// 4096-entry codon table in shared memory, ~55 instructions per four amino acids instead of ~100) and the
// table-per-byte path of k3_lane for a group that holds anything else.
#define K34_AGG 512                 // block-level count combine: direct-mapped, first come first served
#define K34_PROBES 16               // longer probe chains are left to k4_insert

struct Key34Tables {
    Key3Tables k3;
    uint8_t codon[4096];            // tf_codon_entry
    uint32_t agg_slot[K34_AGG];
    uint32_t agg_cnt[K34_AGG];
};

// four amino acids of a group that holds a byte other than a canonical base: the per-byte tables (rare; out of line).
// One copy per UMI mode: a copy called from one kernel only lets that kernel's tables stay where the compiler put them
// before UMIs existed.
template <bool UMI>
__device__ __noinline__ uint32_t k34_group_slow(const Key3Tables *K, uint32_t x0, uint32_t x1, uint32_t x2)
{
    const uint32_t i0 = K->lut25[x0 & 0xFFu] + K->lut5[(x0 >> 8) & 0xFFu] + K->lut1[(x0 >> 16) & 0xFFu];
    const uint32_t i1 = K->lut25[x0 >> 24] + K->lut5[x1 & 0xFFu] + K->lut1[(x1 >> 8) & 0xFFu];
    const uint32_t i2 = K->lut25[(x1 >> 16) & 0xFFu] + K->lut5[x1 >> 24] + K->lut1[x2 & 0xFFu];
    const uint32_t i3 = K->lut25[(x2 >> 8) & 0xFFu] + K->lut5[(x2 >> 16) & 0xFFu] + K->lut1[x2 >> 24];
    return (uint32_t)K->aa[i0] | ((uint32_t)K->aa[i1] << 8) | ((uint32_t)K->aa[i2] << 16) | ((uint32_t)K->aa[i3] << 24);
}

// twelve bases -> four amino acids (codon a = bytes 3a .. 3a+2 of the 12; translate, src/lib.rs:16-44)
template <bool UMI>
__device__ __forceinline__ uint32_t k34_group(const Key34Tables &T, uint32_t x0, uint32_t x1, uint32_t x2)
{
    uint32_t i0, i1, i2, i3;
    if (tf_codons12(x0, x1, x2, i0, i1, i2, i3))
        return (uint32_t)T.codon[i0] | ((uint32_t)T.codon[i1] << 8) | ((uint32_t)T.codon[i2] << 16) | ((uint32_t)T.codon[i3] << 24);
    return k34_group_slow<UMI>(&T.k3, x0, x1, x2);
}

// The common case: region in the shared-memory tile, key block in shared memory, at most 32 key words.  The loop
// has no branch (four groups are in flight per lane): a group that holds anything but canonical bases only sets its
// bit, and those groups are redone through the per-byte tables afterwards, with the hash corrected by the difference.
// The last word (1..4 amino acids, masked) is peeled off the loop.
__device__ __forceinline__ uint32_t k34_group_fast(const Key34Tables &T, uint32_t x0, uint32_t x1, uint32_t x2, bool &ok)
{
    uint32_t i0, i1, i2, i3;
    ok = tf_codons12(x0, x1, x2, i0, i1, i2, i3);           // the indices stay below 4096 whatever the bytes are
    return (uint32_t)T.codon[i0] | ((uint32_t)T.codon[i1] << 8) | ((uint32_t)T.codon[i2] << 16) | ((uint32_t)T.codon[i3] << 24);
}

template <bool UMI>
__device__ __forceinline__ uint64_t k34_lane_hot(const Key34Tables &T, const uint32_t *w, uint32_t sh, uint32_t kl, uint32_t *out)
{
    const uint32_t nw = (kl + 3) >> 2, npad = ((kl + 15u) & ~15u) >> 2;
    uint64_t acc = 0;
    uint32_t bad = 0;                                      // bit wi: group wi must be redone
    uint32_t t0 = w[0];
    const uint32_t *p = w + 1;
    uint32_t wi = 0;
#pragma unroll 4
    for (; wi + 1 < nw; ++wi) {
        const uint32_t t1 = p[0], t2 = p[1], t3 = p[2];
        p += 3;
        bool ok;
        const uint32_t word = k34_group_fast(T, __funnelshift_r(t0, t1, sh), __funnelshift_r(t1, t2, sh), __funnelshift_r(t2, t3, sh), ok);
        t0 = t3;
        bad |= (ok ? 0u : 1u) << wi;
        acc += (uint64_t)(word ^ VFB_HASH_K) * T.k3.mult[wi];
        out[wi] = word;
    }
    const uint32_t left = kl - 4 * wi;                     // 1..4 key bytes in the last word
    const uint32_t last_mask = left < 4 ? (1u << (8 * left)) - 1u : 0xFFFFFFFFu;
    {
        const uint32_t t1 = p[0], t2 = p[1], t3 = p[2];
        bool ok;
        const uint32_t word = k34_group_fast(T, __funnelshift_r(t0, t1, sh), __funnelshift_r(t1, t2, sh), __funnelshift_r(t2, t3, sh), ok) & last_mask;
        bad |= (ok ? 0u : 1u) << wi;
        acc += (uint64_t)(word ^ VFB_HASH_K) * T.k3.mult[wi];
        out[wi] = word;
    }
    for (wi = nw; wi < npad; ++wi) out[wi] = 0u;
    while (bad) {
        const uint32_t g = (uint32_t)__ffs((int)bad) - 1u;
        bad &= bad - 1u;
        const uint32_t *q = w + 3 * g;
        uint32_t word = k34_group_slow<UMI>(&T.k3, __funnelshift_r(q[0], q[1], sh), __funnelshift_r(q[1], q[2], sh), __funnelshift_r(q[2], q[3], sh));
        if (g + 1 == nw) word &= last_mask;
        const uint32_t was = out[g];
        acc += ((uint64_t)(word ^ VFB_HASH_K) - (uint64_t)(was ^ VFB_HASH_K)) * T.k3.mult[g];
        out[g] = word;
    }
    return acc;
}

// Everything else: regions read from global memory, keys written straight to the batch's key space, long keys.
template <bool SMEM, bool UMI>
__device__ __forceinline__ uint64_t k34_lane_translate(const Key34Tables &T, const uint32_t *w, const uint32_t *limit, uint32_t sh,
                                                       uint32_t kl, uint32_t *out)
{
    const uint32_t nw = (kl + 3) >> 2, npad = ((kl + 15u) & ~15u) >> 2;
    uint64_t acc = 0;
    uint32_t t0 = k3_word<SMEM>(w, 0, limit), wp = 1;
    for (uint32_t wi = 0; wi < nw; ++wi) {
        const uint32_t t1 = k3_word<SMEM>(w, wp, limit), t2 = k3_word<SMEM>(w, wp + 1, limit), t3 = k3_word<SMEM>(w, wp + 2, limit);
        wp += 3;
        uint32_t word = k34_group<UMI>(T, __funnelshift_r(t0, t1, sh), __funnelshift_r(t1, t2, sh), __funnelshift_r(t2, t3, sh));
        t0 = t3;
        const uint32_t left = kl - 4 * wi;                 // key bytes from this word on, >= 1
        if (left < 4) word &= (1u << (8 * left)) - 1u;
        acc += (uint64_t)(word ^ VFB_HASH_K) * (wi < KEY_MULTS ? T.k3.mult[wi] : vfb_hash_mult(wi));
        out[wi] = word;
    }
    for (uint32_t wi = nw; wi < npad; ++wi) out[wi] = 0u;
    return acc;
}

// The slot of the published row that holds `key` (klen bytes, zero-padded to 16), or VFB_NONE.
__device__ __forceinline__ uint32_t k34_probe(const DevTable &t, uint64_t h, uint32_t klen, const uint4 *key)
{
    const uint32_t tag = (uint32_t)(h >> 32);
    const uint64_t mask = t.capacity - 1;
    uint64_t slot = h & mask;
    const uint32_t n16 = (klen + 15u) >> 4;
#pragma unroll 1
    for (int tries = 0; tries < K34_PROBES; ++tries) {
        const ulonglong2 *ent = reinterpret_cast<const ulonglong2 *>(t.slots + slot * VFB_SLOT_WORDS);
        const ulonglong2 a = __ldcg(ent), b = __ldcg(ent + 1);      // one 32-byte sector
        if (a.x == 0ull) return VFB_NONE;
        if ((uint32_t)(a.x >> 32) == tag && !((uint32_t)a.x & REF_BATCH) && (uint32_t)b.y == klen) {
            const uint4 *row = reinterpret_cast<const uint4 *>(t.arena + b.x);
            uint32_t diff = 0;
            uint32_t c = 0;
            for (; c + 4 <= n16; c += 4) {             // the loads of a key are in flight together
                uint4 u[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) u[k] = __ldcg(row + c + k);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const uint4 v = key[c + k];
                    diff |= (u[k].x ^ v.x) | (u[k].y ^ v.y) | (u[k].z ^ v.z) | (u[k].w ^ v.w);
                }
            }
            for (; c < n16; ++c) {
                const uint4 u = __ldcg(row + c), v = key[c];
                diff |= (u.x ^ v.x) | (u.y ^ v.y) | (u.z ^ v.z) | (u.w ^ v.w);
            }
            if (diff == 0u) return (uint32_t)slot;
        }
        slot = (slot + 1) & mask;
    }
    return VFB_NONE;
}

// ---- the warp's software pipeline
// A warp's unit (32 reads) goes through three steps, one loop iteration apart, so that no step waits for memory
// it has only just asked for (the kernel runs about ten warps per SM — the tiles take the shared memory — which
// is far too few to hide two dependent DRAM round trips per read behind other warps):
//   iteration i      the unit's text tile (bulk copy issued during iteration i-1) is translated into key block
//                    i % 3, keys are hashed, and every lane asks for its key's home slot (cp.async, 32 bytes
//                    into a per-lane landing zone);
//   iteration i+1    the slot has landed: empty or another key's -> the read is left to the insert kernels; tag and
//                    length match a published row -> the lane asks for that row's key bytes from the arena
//                    (cp.async, at most K34_ROW_BYTES);
//   iteration i+2    the row's key has landed: equal to the lane's key (still in key block i % 3) -> counted here;
//                    otherwise the read joins the list for the insert kernels, which settle collisions exactly.
// Only the home slot is looked at; keys that sit further down a probe chain simply take the insert kernels.
// Lanes the pipeline cannot take (keys longer than K34_ROW_BYTES, units whose keys do not fit the key block) probe
// synchronously (k34_probe).
#define K34_ROW_BYTES 80
#define K34_STAGE_BYTES (32 * 32 + 32 * K34_ROW_BYTES)      // per warp: slot and row landing zones

__device__ __forceinline__ void k34_cp16(uint32_t smem_dst, const void *src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(src) : "memory");
}

// Count a read whose key lives in `slot`: combined per block for the slots that got an entry of the block's small
// direct-mapped table (popular variants), straight to the table otherwise.
__device__ __forceinline__ void k34_count_hit(Key34Tables &T, const DevTable &tab, uint32_t slot)
{
    const uint32_t e = (slot * 2654435761u) >> 23;          // K34_AGG = 512 entries
    uint32_t cur = *reinterpret_cast<volatile uint32_t *>(&T.agg_slot[e]);
    if (cur == VFB_NONE) {
        cur = atomicCAS(&T.agg_slot[e], VFB_NONE, slot);
        if (cur == VFB_NONE) cur = slot;
    }
    if (cur == slot) atomicAdd(&T.agg_cnt[e], 1u);
    else atomicAdd(&tab.slots[(uint64_t)slot * VFB_SLOT_WORDS + 1], 1ull);
}

// The lanes with `miss` set append their keys to the compact list for the insert kernels.  copy_key: the key is in
// shared memory (`key`) and gets key space here; otherwise it already sits at `ko_have` in the batch's key space.
// Called by the whole warp.
__device__ __forceinline__ void k34_emit_misses(const KeyJob &job, uint32_t *n_miss, bool miss, bool copy_key, const uint32_t *key,
                                                unsigned long long ko_have, uint32_t klen, uint64_t h)
{
    const int lane = threadIdx.x & 31;
    const unsigned missing = __ballot_sync(0xffffffffu, miss);
    if (!missing) return;
    const uint32_t padded = (klen + 15u) & ~15u;
    uint32_t m_incl = (miss && copy_key) ? padded : 0u;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, m_incl, o);
        if (lane >= o) m_incl += t;
    }
    const uint32_t m_total = __shfl_sync(0xffffffffu, m_incl, 31);
    uint32_t m0 = 0;
    unsigned long long m_base = 0;
    if (lane == 0) m0 = atomicAdd(n_miss, (uint32_t)__popc(missing));
    if (lane == 31 && m_total) m_base = atomicAdd(job.key_cursor, (unsigned long long)m_total);
    m0 = __shfl_sync(0xffffffffu, m0, 0);
    m_base = __shfl_sync(0xffffffffu, m_base, 31);
    if (miss) {
        const uint32_t m = m0 + __popc(missing & ((1u << lane) - 1u));
        unsigned long long ko = ko_have;
        if (copy_key) {
            ko = m_base + (m_incl - padded);
            const uint4 *src = reinterpret_cast<const uint4 *>(key);
            uint4 *dst = reinterpret_cast<uint4 *>(job.keys + ko);
            for (uint32_t c = 0; c < padded / 16; ++c) dst[c] = src[c];
        }
        job.koff[m] = ko;
        job.klen[m] = klen;
        job.khash[m] = h;
    }
}

#define K34_WARPS_MAX 16

template <bool TRANSLATE, bool UMI>
__global__ void __maxnreg__(128)
k34_keys_count(const __grid_constant__ KeyJob job, const __grid_constant__ DevTable tab, uint32_t *n_miss,
               const uint32_t tile_bytes, const uint32_t out_bytes, const __grid_constant__ UmiArgs umi)
{
    extern __shared__ __align__(128) uint8_t dyn[];
    __shared__ Key34Tables T;
    __shared__ unsigned long long bars[K34_WARPS_MAX];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        const uint32_t c = i >= 128 ? 4u : tr_index((uint8_t)i);
        T.k3.lut25[i] = (uint8_t)(25u * c); T.k3.lut5[i] = (uint8_t)(5u * c); T.k3.lut1[i] = (uint8_t)c;
    }
    for (int i = threadIdx.x; i < 128; i += blockDim.x) {
        const int c0 = i / 25, c1 = (i / 5) % 5, c2 = i % 5;
        T.k3.aa[i] = (i >= 125 || c0 == 4 || c1 == 4 || c2 == 4) ? (uint8_t)'X' : (uint8_t)c_aa[c0 * 16 + c1 * 4 + c2];
    }
    for (int i = threadIdx.x; i < KEY_MULTS; i += blockDim.x) T.k3.mult[i] = vfb_hash_mult((uint32_t)i);
    for (int i = threadIdx.x; i < 4096; i += blockDim.x) T.codon[i] = tf_codon_entry((uint32_t)i, c_aa);
    for (int i = threadIdx.x; i < K34_AGG; i += blockDim.x) { T.agg_slot[i] = VFB_NONE; T.agg_cnt[i] = 0u; }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    if (lane == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(k3_smem_u32(bars + warp)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    // per warp: text tile | three key blocks | slot landing zone (32 B per lane) | row landing zone
    const size_t per_warp = (size_t)tile_bytes + K3T_SLACK + 3 * (size_t)out_bytes + K34_STAGE_BYTES;
    uint8_t *tile = dyn + (size_t)warp * per_warp;
    const uint32_t *tile32 = reinterpret_cast<const uint32_t *>(tile);
    uint8_t *ring = tile + tile_bytes + K3T_SLACK;
    uint8_t *slot_land = ring + 3 * (size_t)out_bytes + (size_t)lane * 32;
    uint8_t *row_land = ring + 3 * (size_t)out_bytes + 32 * 32 + (size_t)lane * K34_ROW_BYTES;
    const uint32_t bar = k3_smem_u32(bars + warp), tile_s = k3_smem_u32(tile);
    const uint32_t slot_land_s = k3_smem_u32(slot_land), row_land_s = k3_smem_u32(row_land);
    const uint64_t mask = tab.capacity - 1;
    uint32_t parity = 0;
    uint32_t my_hits = 0;                                  // reads this lane counted
    uint32_t my_short = 0;                                 // UMI: reads of this lane whose UMI does not fit
    const uint32_t n_units = (job.n_reads + 31) / 32;
    const uint32_t stride = gridDim.x * n_warps;

    // what a lane knows about its read of a unit before the text is there
    struct Plan {
        uint32_t klen, V, roff;        // key length (0 = no key), region length, region offset in the text
        uint32_t lo, n_bytes, lead;    // the unit's tile: first region byte, bytes to stage, misalignment of lo
        bool owners, staged;
    };
    auto make_plan = [&](bool in_range, uint32_t s, uint32_t e, vfb_span sp) {
        Plan p;
        p.klen = 0; p.V = 0; p.roff = 0;
        // src/lib.rs:288: both located and start < end (strict)
        if (in_range && s != VFB_NONE && e != VFB_NONE && s < e && e <= sp.len) {
            p.V = e - s;
            p.roff = sp.off + s;
            if (!TRANSLATE) p.klen = p.V;
            else if (p.V % 3 == 0) p.klen = p.V / 3;                  // :17-19 partial codon -> None
        }
        p.owners = __ballot_sync(0xffffffffu, p.klen != 0) != 0;
        p.lo = __reduce_min_sync(0xffffffffu, p.klen ? p.roff : 0xFFFFFFFFu);
        const uint32_t last = __reduce_max_sync(0xffffffffu, p.klen ? p.roff + (p.V - 1) : 0u);
        p.lead = (uint32_t)(reinterpret_cast<uintptr_t>(job.text + p.lo) & 15u);
        const uint64_t nb = ((uint64_t)(last - p.lo) + 1 + p.lead + 15) & ~15ull;
        p.staged = p.owners && nb <= tile_bytes;
        p.n_bytes = (uint32_t)nb;
        return p;
    };
    auto issue_tile = [&](const Plan &p) {
        if (p.staged && lane == 0) {
            const uintptr_t g0 = reinterpret_cast<uintptr_t>(job.text + p.lo);
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(p.n_bytes) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(tile_s), "l"(g0 & ~(uintptr_t)15), "r"(p.n_bytes), "r"(bar) : "memory");
        }
    };

    uint32_t unit = blockIdx.x * n_warps + warp;
    Plan cur;
    // UMI: where the current / next unit's UMIs sit (the plans' klen include them; a unit's tile still covers the
    // regions of reads whose UMI does not fit)
    uint32_t cur_uoff = 0, nxt_uoff = 0;
    {
        const uint32_t r = unit * 32 + lane;
        const bool in = unit < n_units && r < job.n_reads;
        uint32_t s = VFB_NONE, e = VFB_NONE;
        vfb_span sp; sp.off = 0; sp.len = 0;
        if (in) { s = job.start[r]; e = job.end[r]; sp = job.spans[r]; }
        cur = make_plan(in, s, e, sp);
        if constexpr (UMI) umi_plan<TRANSLATE>(umi, job, sp, cur.roff, cur.V, cur.klen, cur_uoff, my_short);
        issue_tile(cur);
    }
    // pipeline registers: p1 = the previous unit (slot asked for), p2 = the one before (row asked for)
    uint64_t h1 = 0, h2 = 0;
    uint32_t klen1 = 0, klen2 = 0, kpos1 = 0, kpos2 = 0;   // kpos: byte offset of the lane's key in the ring
    uint32_t st1 = 0, st2 = 0;                             // p1: 1 = slot on its way; p2: 1 = miss, 2 = row on its way
    uint32_t slot2 = 0;
    unsigned rsv_mask = 0;                                 // p2 lanes whose list entry and key space are already claimed
    uint32_t rsv_m0 = 0, rsv_rank = 0, rsv_off = 0;
    unsigned long long rsv_base = 0;
    bool any1 = false, any2 = false;                       // warp-uniform: some lane of p1 / p2 is live
    uint32_t bi = 0;                                       // key block of the current unit

    for (;; unit += stride) {
        const bool live = unit < n_units;
        if (!live && !any1 && !any2) break;
        __syncwarp();                                      // key block `bi` is free: its previous unit left the pipeline
        // ---- the next unit's boundaries and span: asked for now, needed after the translate
        uint32_t ns = VFB_NONE, ne = VFB_NONE;
        vfb_span nsp; nsp.off = 0; nsp.len = 0;
        const uint32_t nr = (unit + stride) * 32 + lane;
        const bool n_in = live && unit + stride < n_units && nr < job.n_reads;
        if (n_in) { ns = job.start[nr]; ne = job.end[nr]; nsp = job.spans[nr]; }

        // ---- this unit: key block layout, translate, hash
        uint32_t klen = live ? cur.klen : 0u;
        const bool owners = live && cur.owners;
        uint64_t h = 0;
        uint32_t padded = 0, local = 0;
        bool out_staged = true;
        unsigned long long base = 0;
        uint32_t *out = nullptr;
        if (owners) {
            padded = (klen + 15u) & ~15u;
            uint32_t incl = padded;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
            local = incl - padded;                         // this lane's key inside the unit's key block
            // keys are assembled in shared memory when the unit's keys fit a key block; otherwise every key of the
            // unit goes to the batch's key space first (claimed here) and is probed from there
            out_staged = total <= out_bytes;
            if (!out_staged) {
                if (lane == 31) base = atomicAdd(job.key_cursor, (unsigned long long)total);
                base = __shfl_sync(0xffffffffu, base, 31);
            }
            uint32_t *blk = reinterpret_cast<uint32_t *>(ring + (size_t)bi * out_bytes);
            out = out_staged ? blk + (local >> 2) : reinterpret_cast<uint32_t *>(job.keys + base + local);
            if (cur.staged) {
                uint32_t ok;
                do {
                    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
                } while (!ok);
                parity ^= 1u;
            }
            if (klen) {
                uint64_t acc;
                uint32_t high = 0;
                const uint32_t kr = UMI ? klen - umi.len : klen;      // the region's part of the key
                if (cur.staged) {
                    const uint32_t toff = cur.lead + (cur.roff - cur.lo);
                    if (TRANSLATE && out_staged && kr <= 128u)
                        acc = k34_lane_hot<UMI>(T, tile32 + (toff >> 2), (toff & 3u) * 8u, kr, blk + (local >> 2));
                    else if (TRANSLATE) acc = k34_lane_translate<true, UMI>(T, tile32 + (toff >> 2), nullptr, (toff & 3u) * 8u, kr, out);
                    else acc = k3_lane<true, false>(T.k3, tile32 + (toff >> 2), nullptr, (toff & 3u) * 8u, kr, out, high);
                } else {
                    const uintptr_t va = reinterpret_cast<uintptr_t>(job.text + cur.roff);
                    const uint32_t *limit = reinterpret_cast<const uint32_t *>((va + cur.V + 3) & ~(uintptr_t)3);
                    const uint32_t *w = reinterpret_cast<const uint32_t *>(va & ~(uintptr_t)3);
                    if (TRANSLATE) acc = k34_lane_translate<false, UMI>(T, w, limit, (uint32_t)(va & 3u) * 8u, kr, out);
                    else acc = k3_lane<false, false>(T.k3, w, limit, (uint32_t)(va & 3u) * 8u, kr, out, high);
                }
                if constexpr (UMI) umi_append(job.text + cur_uoff, umi.len, kr, out, acc, T.k3.mult);
                h = vfb_hash_finish(acc, klen);
                if (job.hash_bits > 0 && job.hash_bits < 64) h &= (1ull << job.hash_bits) - 1;
                // String::from_utf8 (:295): only regions holding a byte >= 0x80 need the validator
                if (!TRANSLATE && high && !utf8_valid(job.text + cur.roff, cur.V)) klen = 0;
            }
        }
        __syncwarp();                                      // the tile has been read by every lane
        // ---- the next unit's tile starts its journey now
        Plan nxt = make_plan(n_in, ns, ne, nsp);
        if constexpr (UMI) umi_plan<TRANSLATE>(umi, job, nsp, nxt.roff, nxt.V, nxt.klen, nxt_uoff, my_short);
        issue_tile(nxt);

        // ---- what was asked for an iteration ago has landed
        asm volatile("cp.async.wait_all;" ::: "memory");
        // p2: compare the row's key with the lane's key; count or hand over
        if (any2) {
            const uint32_t *key2 = reinterpret_cast<const uint32_t *>(ring + kpos2);
            bool late = false;                             // tag and length matched, the key does not (a full hash collision)
            if (st2 == 2u) {
                const uint4 *row = reinterpret_cast<const uint4 *>(row_land);
                const uint4 *key = reinterpret_cast<const uint4 *>(key2);
                const uint32_t n16 = (klen2 + 15u) >> 4;
                uint32_t diff = 0;
#pragma unroll
                for (uint32_t c = 0; c < K34_ROW_BYTES / 16; ++c)
                    if (c < n16) {
                        const uint4 u = row[c], v = key[c];
                        diff |= (u.x ^ v.x) | (u.y ^ v.y) | (u.z ^ v.z) | (u.w ^ v.w);
                    }
                if (diff == 0u) { ++my_hits; k34_count_hit(T, tab, slot2); }
                else late = true;
            }
            // reads that were certain to go to the insert kernels an iteration ago: their list entries and key space
            // were claimed then, the claims' results are first looked at here
            if (rsv_mask) {
                const uint32_t m0 = __shfl_sync(0xffffffffu, rsv_m0, 0);
                const unsigned long long mb = __shfl_sync(0xffffffffu, rsv_base, 31);
                if (st2 == 1u) {
                    const uint32_t m = m0 + rsv_rank;
                    const unsigned long long ko = mb + rsv_off;
                    const uint4 *src = reinterpret_cast<const uint4 *>(key2);
                    uint4 *dst = reinterpret_cast<uint4 *>(job.keys + ko);
                    const uint32_t n16 = (klen2 + 15u) >> 4;
                    for (uint32_t c = 0; c < n16; ++c) dst[c] = src[c];
                    job.koff[m] = ko;
                    job.klen[m] = klen2;
                    job.khash[m] = h2;
                }
            }
            k34_emit_misses(job, n_miss, late, true, key2, 0ull, klen2, h2);
        }
        // p1: look at the slot; ask for the row's key, or claim a list entry and key space for the insert kernels
        st2 = 0;
        rsv_mask = 0;
        if (any1) {
            if (st1) {
                const ulonglong2 a = *reinterpret_cast<const ulonglong2 *>(slot_land);
                const ulonglong2 b = *reinterpret_cast<const ulonglong2 *>(slot_land + 16);
                st2 = 1u;                                  // empty, another key, or not a published row: the insert kernels
                if (a.x != 0ull && (uint32_t)(a.x >> 32) == (uint32_t)(h1 >> 32) && !((uint32_t)a.x & REF_BATCH) &&
                    (uint32_t)b.y == klen1) {
                    st2 = 2u;
                    const uint8_t *row = tab.arena + b.x;
                    const uint32_t n16 = (klen1 + 15u) >> 4;
#pragma unroll
                    for (uint32_t c = 0; c < K34_ROW_BYTES / 16; ++c)
                        if (c < n16) k34_cp16(row_land_s + 16 * c, row + 16 * c);
                }
            }
            rsv_mask = __ballot_sync(0xffffffffu, st2 == 1u);
            if (rsv_mask) {
                // the two claims are single addresses for the whole grid: their answers are not waited for here
                const uint32_t padded1 = (klen1 + 15u) & ~15u;
                uint32_t mi = st2 == 1u ? padded1 : 0u;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t t = __shfl_up_sync(0xffffffffu, mi, o);
                    if (lane >= o) mi += t;
                }
                // (predicated atomics written straight into the loop-carried registers: a compiler-made copy of the
                // result would wait for it here)
                asm volatile("{\n.reg .pred p;\nsetp.eq.u32 p, %2, 0;\n@p atom.global.add.u32 %0, [%1], %3;\n}"
                             : "+r"(rsv_m0) : "l"(n_miss), "r"(lane), "r"((uint32_t)__popc(rsv_mask)) : "memory");
                asm volatile("{\n.reg .pred p;\nsetp.eq.u32 p, %2, 31;\n@p atom.global.add.u64 %0, [%1], %3;\n}"
                             : "+l"(rsv_base) : "l"(job.key_cursor), "r"(lane), "l"((unsigned long long)mi) : "memory");
                rsv_rank = (uint32_t)__popc(rsv_mask & ((1u << lane) - 1u));
                rsv_off = mi - padded1;
            }
            h2 = h1; klen2 = klen1; kpos2 = kpos1; slot2 = (uint32_t)(h1 & mask);
        }
        any2 = any1;
        // p0 -> p1: ask for the home slot, or (lanes the pipeline cannot take) probe synchronously
        st1 = 0;
        any1 = false;
        if (owners) {
            const bool piped = klen != 0 && out_staged && padded <= K34_ROW_BYTES;
            if (piped) {
                const unsigned long long *ent = tab.slots + (h & mask) * VFB_SLOT_WORDS;
                k34_cp16(slot_land_s, ent);
                k34_cp16(slot_land_s + 16, ent + 2);
                st1 = 1u;
                h1 = h; klen1 = klen; kpos1 = bi * out_bytes + local;
            }
            any1 = __ballot_sync(0xffffffffu, piped) != 0;
            const bool direct = klen != 0 && !piped;
            if (__ballot_sync(0xffffffffu, direct)) {
                bool miss = false;
                if (direct) {
                    const uint32_t slot = k34_probe(tab, h, klen, reinterpret_cast<const uint4 *>(out));
                    if (slot != VFB_NONE) { ++my_hits; k34_count_hit(T, tab, slot); }
                    else miss = true;
                }
                k34_emit_misses(job, n_miss, miss, out_staged, out, base + local, klen, h);
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        cur = nxt;
        if constexpr (UMI) cur_uoff = nxt_uoff;
        bi = bi == 2u ? 0u : bi + 1u;
    }
    // ---- reads counted by this warp, block-level counts
    {
        uint32_t hits = my_hits;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) hits += __shfl_xor_sync(0xffffffffu, hits, o);
        if (lane == 0 && hits) {
            atomicAdd(&tab.counters[2], (unsigned long long)hits);
            atomicAdd(&tab.counters[3], (unsigned long long)hits);
        }
    }
    if constexpr (UMI) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) my_short += __shfl_xor_sync(0xffffffffu, my_short, o);
        if (lane == 0 && my_short) atomicAdd(umi.n_short, (unsigned long long)my_short);
    }
    __syncthreads();
    for (int e = threadIdx.x; e < K34_AGG; e += blockDim.x)
        if (T.agg_slot[e] != VFB_NONE && T.agg_cnt[e])
            atomicAdd(&tab.slots[(uint64_t)T.agg_slot[e] * VFB_SLOT_WORDS + 1], (unsigned long long)T.agg_cnt[e]);
}

template <bool TRANSLATE, bool UMI>
static int launch_keys_count_t(const KeyJob &job, const DevTable &tab, uint32_t *n_miss, cudaStream_t st, const UmiArgs &umi)
{
    const uint32_t tile = vfb_tile_bytes_for(job.text_bytes, job.n_reads);
    // a key block holds the 32 keys of a unit at their expected length (a third of what the adapters leave of the
    // read for amino acids, plus the UMI)
    const uint64_t stride = job.n_reads ? job.text_bytes / job.n_reads : 0;
    const uint64_t region_ub = stride > job.flank_bytes ? stride - job.flank_bytes : 0;
    const uint64_t key_ub = (TRANSLATE ? region_ub / 3 : region_ub) + umi.len;
    uint32_t out_bytes = (uint32_t)(32 * ((key_ub + 15) & ~15ull));
    if (out_bytes < 1024) out_bytes = 1024;
    if (out_bytes > 4096u) out_bytes = 4096u;
    const size_t per_warp = (size_t)tile + K3T_SLACK + 3 * (size_t)out_bytes + K34_STAGE_BYTES;
    // as many warps per SM as the shared memory allows; the tables are per block, so few large blocks
    int best_w = 0, best_total = 0;
    for (int w = K34_WARPS_MAX; w >= 1; --w) {
        const size_t per_block = (size_t)w * per_warp + sizeof(Key34Tables) + 8 * K34_WARPS_MAX + 1024;
        int bps = (int)(VFB_SMEM_BLOCK_MAX / per_block);
        if (bps * w > 16) bps = 16 / w;               // 128 registers per thread: 16 warps fit the register file
        if (bps * w > best_total) { best_total = bps * w; best_w = w; }
    }
    if (best_total == 0) return -1;
    const size_t smem = (size_t)best_w * per_warp;
    VFB_CUDA(cudaFuncSetAttribute(k34_keys_count<TRANSLATE, UMI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const uint32_t units = (job.n_reads + 31) / 32;
    uint32_t blocks = (units + best_w - 1) / best_w;
    const uint32_t cap = 148u * (uint32_t)(best_total / best_w);
    if (blocks > cap) blocks = cap;
    k34_keys_count<TRANSLATE, UMI><<<blocks, best_w * 32, smem, st>>>(job, tab, n_miss, tile, out_bytes, umi);
    return VFB_OK;
}

// Fused key + count launch: afterwards *n_miss keys sit in job.koff / klen / khash (compact) for launch_insert.
// Returns -1 when the tile kernel does not apply (the caller then runs launch_keys + launch_insert over all reads).
int launch_keys_count(const KeyJob &job, const DevTable &tab, uint32_t *n_miss, cudaStream_t st, const UmiArgs &umi)
{
    if (job.n_reads == 0 || job.text_bytes == 0) return -1;
    int rc;
    if (!umi.len) rc = job.skip_translation ? launch_keys_count_t<false, false>(job, tab, n_miss, st, umi)
                                            : launch_keys_count_t<true, false>(job, tab, n_miss, st, umi);
    else rc = job.skip_translation ? launch_keys_count_t<false, true>(job, tab, n_miss, st, umi)
                                   : launch_keys_count_t<true, true>(job, tab, n_miss, st, umi);
    if (rc != VFB_OK) return rc;
    ++g_launches;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

// One thread per key: probe, claim or match (full key compare), count.  Counts are first
// combined per block in a small shared-memory table keyed by slot, so a popular variant costs
// one global atomic per block instead of one per read (same-address atomics serialise in L2).
#define INS_THREADS 256
#define INS_AGG 512

__global__ void __launch_bounds__(INS_THREADS)
k4_insert(const __grid_constant__ InsertArgs a)
{
    __shared__ uint32_t agg_slot[INS_AGG];
    __shared__ unsigned long long agg_cnt[INS_AGG];
    const InsertJob &j = a.job;
    const DevTable &t = a.t;
    // the key list may have been compacted on the device (k34_keys_count): its length is then a device word
    uint32_t n_keys = j.n_keys;
    if (j.n_keys_dev) { const uint32_t nd = *j.n_keys_dev; n_keys = nd < n_keys ? nd : n_keys; }
    const uint32_t n_blk = (n_keys + INS_THREADS - 1) / INS_THREADS;
    // blocks take 256 keys at a time; the shared count table is per 256 keys (it can never fill up)
    for (uint32_t blk = blockIdx.x; blk < n_blk; blk += gridDim.x) {
    for (int e = threadIdx.x; e < INS_AGG; e += INS_THREADS) { agg_slot[e] = VFB_NONE; agg_cnt[e] = 0ull; }
    __syncthreads();

    const uint32_t i = blk * INS_THREADS + threadIdx.x;
    uint32_t klen = 0;
    if (i < n_keys) klen = j.klen[i];
    const unsigned active = __ballot_sync(0xffffffffu, klen != 0);
    if (active) {
        // reads counted by this warp: one atomic per warp
        unsigned long long add = klen ? (j.kcount ? j.kcount[i] : 1ull) : 0ull;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) add += __shfl_xor_sync(0xffffffffu, add, o);
        if ((threadIdx.x & 31) == 0 && add) atomicAdd(&t.counters[2], add);
    }
    uint32_t owner = VFB_NONE;
    if (klen) {
        const uint64_t h = j.khash[i];
        const unsigned long long cnt = j.kcount ? j.kcount[i] : 1ull;
        const uint32_t tag = (uint32_t)(h >> 32);
        const uint64_t mask = t.capacity - 1;
        uint64_t slot = h & mask;
        const unsigned long long mine = ((unsigned long long)tag << 32) | REF_BATCH | i;
        const uint8_t *mykey = job_key(j, i);
        for (;;) {
            unsigned long long *ent = t.slots + slot * VFB_SLOT_WORDS;
            // the whole 32-byte slot in one go (two 16-byte loads of one sector, L1 bypassed): a row's
            // arena offset and length are there when the tag matches, no second round trip
            unsigned long long cur, cnt_unused, m_off, m_len;
            asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(cur), "=l"(cnt_unused) : "l"(ent) : "memory");
            asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(m_off), "=l"(m_len) : "l"(ent + 2) : "memory");
            (void)cnt_unused;
            if (cur == 0ull) {
                cur = atomicCAS(ent, 0ull, mine);
                if (cur == 0ull) {
                    owner = (uint32_t)slot;
                    break;
                }
            }
            if ((uint32_t)(cur >> 32) == tag) {
                const uint32_t ref = (uint32_t)cur;
                const uint8_t *okey;
                uint32_t olen;
                if (ref & REF_BATCH) {
                    const uint32_t o = ref & ~REF_BATCH;
                    okey = job_key(j, o);
                    olen = j.klen[o];
                } else {
                    // a row published by an earlier batch: its arena offset and length sit in the slot
                    okey = t.arena + m_off;
                    olen = (uint32_t)m_len;
                }
                if (olen == klen && keys_equal16(okey, mykey, klen)) break;
            }
            slot = (slot + 1) & mask;
        }
        // block-level combine: claim (or find) this slot's entry in the shared table
        const uint32_t s32 = (uint32_t)slot;
        uint32_t e = (s32 * 2654435761u) >> 23;
        for (;;) {
            const uint32_t old = atomicCAS(&agg_slot[e], VFB_NONE, s32);
            if (old == VFB_NONE || old == s32) { atomicAdd(&agg_cnt[e], cnt); break; }
            e = (e + 1) & (INS_AGG - 1);
        }
    }
    if (i < n_keys) j.owner_slot[i] = owner;
    __syncthreads();
    for (int e = threadIdx.x; e < INS_AGG; e += INS_THREADS)
        if (agg_slot[e] != VFB_NONE) atomicAdd(&t.slots[(uint64_t)agg_slot[e] * VFB_SLOT_WORDS + 1], agg_cnt[e]);
    __syncthreads();
    }
}

// Owners of freshly claimed slots move their key into the arena and turn the slot's
// batch reference into a row reference.  Row ids and arena space are claimed once per warp.
__global__ void __launch_bounds__(256)
k4_publish(const __grid_constant__ InsertArgs a)
{
    const InsertJob &j = a.job;
    const DevTable &t = a.t;
    uint32_t n_keys = j.n_keys;
    if (j.n_keys_dev) { const uint32_t nd = *j.n_keys_dev; n_keys = nd < n_keys ? nd : n_keys; }
    const uint32_t n_blk = (n_keys + 255) / 256;
    const int lane = threadIdx.x & 31;
    // row ids and arena space are claimed once per BLOCK (per 256 keys): the two counters are single addresses,
    // and a claim per warp made every warp of the grid queue up on them
    __shared__ uint32_t s_rows[8], s_bytes[8];
    __shared__ unsigned long long s_row0, s_off0;
    for (uint32_t blk = blockIdx.x; blk < n_blk; blk += gridDim.x) {
        const uint32_t i = blk * 256 + threadIdx.x;
        uint32_t slot = VFB_NONE, klen = 0;
        if (i < n_keys) slot = j.owner_slot[i];
        const bool own = slot != VFB_NONE;
        if (own) klen = j.klen[i];
        const unsigned m = __ballot_sync(0xffffffffu, own);
        const uint32_t padded = own ? (klen + 15u) & ~15u : 0u;
        uint32_t incl = padded;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        const int warp = threadIdx.x >> 5;
        if (lane == 31) { s_rows[warp] = (uint32_t)__popc(m); s_bytes[warp] = incl; }
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t rows = 0, bytes = 0;
            for (int w = 0; w < 8; ++w) {
                const uint32_t rw = s_rows[w], bw = s_bytes[w];
                s_rows[w] = rows; s_bytes[w] = bytes;          // exclusive over the block's warps
                rows += rw; bytes += bw;
            }
            if (rows) {
                s_row0 = atomicAdd(&t.counters[0], (unsigned long long)rows);
                s_off0 = atomicAdd(&t.counters[1], (unsigned long long)bytes);
            }
        }
        __syncthreads();
        const unsigned long long row0 = s_row0 + s_rows[warp], off0 = s_off0 + s_bytes[warp];
        if (own) {
            const unsigned long long row = row0 + __popc(m & ((1u << lane) - 1));
            const unsigned long long off = off0 + (incl - padded);
            const uint4 *src = reinterpret_cast<const uint4 *>(job_key(j, i));
            uint4 *dst = reinterpret_cast<uint4 *>(t.arena + off);
            for (uint32_t c = 0; c < padded / 16; ++c) dst[c] = src[c];
            const uint64_t h = j.khash[i];
            t.row_hash[row] = h;
            t.row_off[row] = off;
            t.row_len[row] = klen;
            t.row_slot[row] = slot;
            unsigned long long *ent = t.slots + (uint64_t)slot * VFB_SLOT_WORDS;
            ent[2] = off;
            ent[3] = klen;
            ent[0] = ((unsigned long long)(uint32_t)(h >> 32) << 32) | (unsigned long long)(row + 1);
        }
        __syncthreads();                                   // s_rows / s_bytes / s_row0 are reused by the next 256 keys
    }
}

int launch_insert(const DevTable &t, const InsertJob &job, cudaStream_t st)
{
    if (job.n_keys == 0) return VFB_OK;
    InsertArgs a;
    a.t = t;
    a.job = job;
    uint32_t blocks = (job.n_keys + 255) / 256;
    // a list whose length only the device knows is walked by resident blocks (most of n_keys may not be there)
    if (job.n_keys_dev && blocks > 148u * 8u) blocks = 148u * 8u;
    k4_insert<<<blocks, 256, 0, st>>>(a);
    k4_publish<<<blocks, 256, 0, st>>>(a);
    g_launches += 2;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

__global__ void __launch_bounds__(256)
k4_rehash(const DevTable o, const DevTable n)
{
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint64_t mask = n.capacity - 1;
    for (uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s < o.capacity; s += stride) {
        const unsigned long long *oe = o.slots + s * VFB_SLOT_WORDS;
        const unsigned long long w = oe[0];
        if (!w) continue;
        const uint32_t row = (uint32_t)w - 1;
        uint64_t slot = o.row_hash[row] & mask;
        for (;;) {
            if (atomicCAS(&n.slots[slot * VFB_SLOT_WORDS], 0ull, w) == 0ull) break;
            slot = (slot + 1) & mask;
        }
        unsigned long long *ne = n.slots + slot * VFB_SLOT_WORDS;
        n.row_slot[row] = (uint32_t)slot;
        ne[1] = oe[1];
        ne[2] = oe[2];
        ne[3] = oe[3];
    }
}

int launch_rehash(const DevTable &old_t, const DevTable &new_t, cudaStream_t st)
{
    uint64_t blocks = (old_t.capacity + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    k4_rehash<<<(uint32_t)blocks, 256, 0, st>>>(old_t, new_t);
    ++g_launches;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

__global__ void __launch_bounds__(256)
k4_export_counts(const DevTable t, uint64_t rows, unsigned long long *row_count)
{
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += stride)
        row_count[r] = t.slots[(uint64_t)t.row_slot[r] * VFB_SLOT_WORDS + 1];
}

int launch_export_counts(const DevTable &t, uint64_t rows, unsigned long long *row_count, cudaStream_t st)
{
    if (rows == 0) return VFB_OK;
    uint64_t blocks = (rows + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    k4_export_counts<<<(uint32_t)blocks, 256, 0, st>>>(t, rows, row_count);
    ++g_launches;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

// ------------------------------------------------------------------------------------ export
// Arrow-style compaction of the table on the device: the rows whose count is not zero (a merge leaves the
// rows it handed to another rank behind with count 0), offsets = exclusive scan of their lengths (plus
// `byte_base`, so that several devices can write consecutive pieces of one column), counts, and the keys
// back to back (the arena pads every key to 16 bytes).
#define EXP_ROWS 1024   // rows per block

template <bool UMI>
__global__ void __launch_bounds__(256)
k_export_sums(const uint32_t *__restrict__ row_len, const unsigned long long *__restrict__ row_count, uint64_t rows,
              unsigned long long *__restrict__ block_bytes, unsigned long long *__restrict__ block_rows, uint32_t trim)
{
    __shared__ unsigned long long s_part[8], s_rows[8];
    const uint64_t r0 = (uint64_t)blockIdx.x * EXP_ROWS;
    unsigned long long acc = 0, kept = 0;
    for (uint32_t k = threadIdx.x; k < EXP_ROWS; k += 256)
        if (r0 + k < rows && row_count[r0 + k]) { acc += row_len[r0 + k] - (UMI ? trim : 0u); ++kept; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        acc += __shfl_xor_sync(0xffffffffu, acc, o);
        kept += __shfl_xor_sync(0xffffffffu, kept, o);
    }
    if ((threadIdx.x & 31) == 0) { s_part[threadIdx.x >> 5] = acc; s_rows[threadIdx.x >> 5] = kept; }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0, n = 0;
        for (int w = 0; w < 8; ++w) { t += s_part[w]; n += s_rows[w]; }
        block_bytes[blockIdx.x] = t;
        block_rows[blockIdx.x] = n;
    }
}

// exclusive scan of the block sums, in place, by one block
__global__ void __launch_bounds__(1024)
k_export_scan(unsigned long long *block_sums, uint64_t n_blocks, unsigned long long *total)
{
    __shared__ unsigned long long s_warp[32];
    __shared__ unsigned long long s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint64_t base = 0; base < n_blocks; base += 1024) {
        const uint64_t i = base + threadIdx.x;
        const unsigned long long v = i < n_blocks ? block_sums[i] : 0ull;
        unsigned long long incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long u = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += u;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            unsigned long long w = s_warp[lane], wi = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long u = __shfl_up_sync(0xffffffffu, wi, o);
                if (lane >= o) wi += u;
            }
            s_warp[lane] = wi - w;      // exclusive over warps
        }
        __syncthreads();
        const unsigned long long carry = s_carry;
        if (i < n_blocks) block_sums[i] = carry + s_warp[warp] + (incl - v);
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = carry + s_warp[warp] + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = s_carry;
}

template <bool UMI>
__global__ void __launch_bounds__(256)
k_export_gather(const DevTable t, uint64_t rows, const unsigned long long *__restrict__ row_count,
                const unsigned long long *__restrict__ block_off, const unsigned long long *__restrict__ block_row,
                unsigned long long byte_base, unsigned long long *__restrict__ offsets,
                unsigned long long *__restrict__ counts, uint8_t *__restrict__ data, uint32_t trim,
                const unsigned long long *__restrict__ row_mol, unsigned long long *__restrict__ molecules)
{
    __shared__ unsigned long long s_off[EXP_ROWS];       // ~0 = row not exported
    __shared__ unsigned long long s_warp[8];
    __shared__ uint32_t s_wrows[8];
    const uint64_t r0 = (uint64_t)blockIdx.x * EXP_ROWS;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // each thread owns 4 consecutive rows of the block
    uint32_t len[4];
    unsigned long long cnt[4];
    unsigned long long mine = 0;
    uint32_t mine_rows = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint64_t r = r0 + threadIdx.x * 4 + k;
        cnt[k] = r < rows ? row_count[r] : 0ull;
        len[k] = cnt[k] ? t.row_len[r] - (UMI ? trim : 0u) : 0u;
        mine += len[k];
        mine_rows += cnt[k] ? 1u : 0u;
    }
    unsigned long long incl = mine;
    uint32_t incl_rows = mine_rows;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long u = __shfl_up_sync(0xffffffffu, incl, o);
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl_rows, o);
        if (lane >= o) { incl += u; incl_rows += v; }
    }
    if (lane == 31) { s_warp[warp] = incl; s_wrows[warp] = incl_rows; }
    __syncthreads();
    unsigned long long wbase = 0;
    uint32_t wrows = 0;
    for (int w = 0; w < warp; ++w) { wbase += s_warp[w]; wrows += s_wrows[w]; }
    unsigned long long o = block_off[blockIdx.x] + wbase + (incl - mine);
    unsigned long long ri = block_row[blockIdx.x] + wrows + (incl_rows - mine_rows);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        s_off[threadIdx.x * 4 + k] = cnt[k] ? o : ~0ull;
        if (cnt[k]) {
            offsets[ri] = byte_base + o;
            counts[ri] = cnt[k];
            if (UMI) molecules[ri] = row_mol[r0 + threadIdx.x * 4 + k];
            ++ri;
        }
        o += len[k];
    }
    __syncthreads();
    // copy: one warp per row, lanes over bytes
    for (uint32_t k = warp; k < EXP_ROWS; k += 8) {
        const uint64_t r = r0 + k;
        if (r >= rows) break;
        if (s_off[k] == ~0ull) continue;
        const uint32_t n = t.row_len[r] - (UMI ? trim : 0u);
        const uint8_t *src = t.arena + t.row_off[r];
        uint8_t *dst = data + s_off[k];
        for (uint32_t b = lane; b < n; b += 32) dst[b] = src[b];
    }
}

// Pass 1: block sums and their scans; totals[0] = key bytes, totals[1] = rows that will be exported.
int launch_export_sizes(const DevTable &t, uint64_t rows, const unsigned long long *row_count,
                        unsigned long long *block_bytes, unsigned long long *block_rows, unsigned long long *totals,
                        cudaStream_t st, uint32_t umi_len)
{
    if (rows == 0) return VFB_OK;
    const uint64_t nb = (rows + EXP_ROWS - 1) / EXP_ROWS;
    if (umi_len) k_export_sums<true><<<(uint32_t)nb, 256, 0, st>>>(t.row_len, row_count, rows, block_bytes, block_rows, umi_len);
    else k_export_sums<false><<<(uint32_t)nb, 256, 0, st>>>(t.row_len, row_count, rows, block_bytes, block_rows, 0);
    k_export_scan<<<1, 1024, 0, st>>>(block_bytes, nb, totals);
    k_export_scan<<<1, 1024, 0, st>>>(block_rows, nb, totals + 1);
    g_launches += 3;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

// Pass 2: offsets[i] = byte_base + start of exported row i, counts[i], keys back to back in data.
int launch_export_gather(const DevTable &t, uint64_t rows, const unsigned long long *row_count,
                         const unsigned long long *block_bytes, const unsigned long long *block_rows,
                         unsigned long long byte_base, unsigned long long *offsets, unsigned long long *counts,
                         uint8_t *data, cudaStream_t st, uint32_t umi_len, const unsigned long long *row_mol,
                         unsigned long long *molecules)
{
    if (rows == 0) return VFB_OK;
    const uint64_t nb = (rows + EXP_ROWS - 1) / EXP_ROWS;
    if (umi_len)
        k_export_gather<true><<<(uint32_t)nb, 256, 0, st>>>(t, rows, row_count, block_bytes, block_rows, byte_base, offsets, counts,
                                                            data, umi_len, row_mol, molecules);
    else
        k_export_gather<false><<<(uint32_t)nb, 256, 0, st>>>(t, rows, row_count, block_bytes, block_rows, byte_base, offsets,
                                                             counts, data, 0, nullptr, nullptr);
    ++g_launches;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

// ------------------------------------------------------------------------------------ merge
// Per warp and per destination part: number of rows, padded key bytes, and this lane's rank /
// byte offset inside its part's group (one atomic per warp per part instead of one per row).
__device__ __forceinline__ void part_group(uint32_t p, bool valid, uint32_t padded, unsigned &peers,
                                           uint32_t &rank, uint32_t &byte_rank, uint32_t &group_bytes)
{
    const int lane = threadIdx.x & 31;
    peers = __match_any_sync(0xffffffffu, valid ? p : 0xFFFFFFFFu);
    rank = __popc(peers & ((1u << lane) - 1));
    byte_rank = 0;
    group_bytes = 0;
    // the shuffles run for every lane (full mask); each lane keeps only its own group's terms
#pragma unroll 1
    for (int l = 0; l < 32; ++l) {
        const uint32_t v = __shfl_sync(0xffffffffu, padded, l);
        if (peers & (1u << l)) {
            group_bytes += v;
            if (l < lane) byte_rank += v;
        }
    }
}

// Rows take part in a merge when their count is not zero and, if `self` names a part (self < n_parts), when
// they are owned by another part: a rank keeps the rows it owns where they are.
// UMI: the owner is that of the variant (the key without its last umi_len bytes); the chunk still carries the full hash.
template <bool UMI>
__device__ __forceinline__ bool part_of(const DevTable &t, uint64_t r, uint32_t n_parts, uint32_t self, uint64_t *h_out,
                                        uint32_t *p_out, unsigned long long **cnt_out, uint32_t umi_len)
{
    const uint64_t h = t.row_hash[r];
    const uint32_t p = vfb_hash_owner(UMI ? vfb_hash_bytes(t.arena + t.row_off[r], t.row_len[r] - umi_len) : h, n_parts);
    *h_out = h;
    *p_out = p;
    if (p == self) return false;
    unsigned long long *cnt = t.slots + (uint64_t)t.row_slot[r] * VFB_SLOT_WORDS + 1;
    *cnt_out = cnt;
    return *cnt != 0ull;
}

template <bool UMI>
__global__ void __launch_bounds__(256)
k5_partition_count(const DevTable t, uint64_t rows, uint32_t n_parts,
                   uint32_t self, unsigned long long *part_rows, unsigned long long *part_keybytes, uint32_t umi_len)
{
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const int lane = threadIdx.x & 31;
    for (uint64_t r0 = (uint64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); r0 < rows; r0 += stride) {
        const uint64_t r = r0 + lane;
        uint64_t h = 0;
        uint32_t p = 0;
        unsigned long long *cnt = nullptr;
        const bool valid = r < rows && part_of<UMI>(t, r, n_parts, self, &h, &p, &cnt, umi_len);
        const uint32_t padded = valid ? (t.row_len[r] + 15u) & ~15u : 0u;
        unsigned peers;
        uint32_t rank, brank, gbytes;
        part_group(p, valid, padded, peers, rank, brank, gbytes);
        if (valid && rank == 0) {
            atomicAdd(&part_rows[p], (unsigned long long)__popc(peers));
            atomicAdd(&part_keybytes[p], (unsigned long long)gbytes);
        }
    }
}

int launch_partition_count(const DevTable &t, uint64_t rows, uint32_t n_parts,
                           uint32_t self, unsigned long long *part_rows, unsigned long long *part_keybytes,
                           cudaStream_t st, uint32_t umi_len)
{
    if (rows == 0) return VFB_OK;
    uint64_t blocks = (rows + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    if (umi_len) k5_partition_count<true><<<(uint32_t)blocks, 256, 0, st>>>(t, rows, n_parts, self, part_rows, part_keybytes, umi_len);
    else k5_partition_count<false><<<(uint32_t)blocks, 256, 0, st>>>(t, rows, n_parts, self, part_rows, part_keybytes, 0);
    ++g_launches;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

// Chunk headers are written by the kernel too (block 0), from the part sizes the count pass left on the device.  An
// export of the whole table (self >= n_parts, vfb_table_partition_fill) gives every part a chunk, an empty one a
// header of zero rows; a keep-own merge sends no chunk for an empty part, and its offset is the next part's.
template <bool UMI>
__global__ void __launch_bounds__(256)
k5_partition_fill(const DevTable t, uint64_t rows, uint32_t n_parts, uint32_t self, bool release,
                  uint8_t *buf, const uint64_t *chunk_off,
                  const uint64_t *part_rows, const uint64_t *part_keybytes,
                  unsigned long long *cursors, uint32_t umi_len)
{
    if (blockIdx.x == 0)
        for (uint32_t p = threadIdx.x; p < n_parts; p += blockDim.x)
            if (p != self && (part_rows[p] || self >= n_parts)) {
                ChunkHeader *hd = reinterpret_cast<ChunkHeader *>(buf + chunk_off[p]);
                hd->magic = VFB_CHUNK_MAGIC; hd->rows = part_rows[p]; hd->key_bytes = part_keybytes[p]; hd->reserved = 0;
            }
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const int lane = threadIdx.x & 31;
    for (uint64_t r0 = (uint64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); r0 < rows; r0 += stride) {
        const uint64_t r = r0 + lane;
        uint64_t h = 0;
        uint32_t p = 0;
        unsigned long long *cnt = nullptr;
        const bool valid = r < rows && part_of<UMI>(t, r, n_parts, self, &h, &p, &cnt, umi_len);
        const uint32_t len = valid ? t.row_len[r] : 0u;
        const uint32_t padded = (len + 15u) & ~15u;
        unsigned peers;
        uint32_t rank, brank, gbytes;
        part_group(p, valid, valid ? padded : 0u, peers, rank, brank, gbytes);
        unsigned long long idx0 = 0, koff0 = 0;
        if (valid && rank == 0) {
            idx0 = atomicAdd(&cursors[2 * p], (unsigned long long)__popc(peers));
            koff0 = atomicAdd(&cursors[2 * p + 1], (unsigned long long)gbytes);
        }
        const int leader = __ffs((int)peers) - 1;
        idx0 = __shfl_sync(0xffffffffu, idx0, leader);
        koff0 = __shfl_sync(0xffffffffu, koff0, leader);
        if (!valid) continue;
        const unsigned long long idx = idx0 + rank, koff = koff0 + brank;
        const uint64_t n = part_rows[p];
        uint8_t *c = buf + chunk_off[p];
        uint64_t *c_hash = reinterpret_cast<uint64_t *>(c + sizeof(ChunkHeader));
        uint64_t *c_count = reinterpret_cast<uint64_t *>(c + sizeof(ChunkHeader) + vfb_align16(n * 8));
        uint64_t *c_koff = reinterpret_cast<uint64_t *>(c + sizeof(ChunkHeader) + vfb_align16(n * 8) * 2);
        uint32_t *c_klen = reinterpret_cast<uint32_t *>(c + sizeof(ChunkHeader) + vfb_align16(n * 8) * 3);
        uint8_t *c_keys = c + sizeof(ChunkHeader) + vfb_align16(n * 8) * 3 + vfb_align16(n * 4);
        c_hash[idx] = h;
        c_count[idx] = *cnt;
        if (release) *cnt = 0ull;            // the count travels with the chunk
        c_koff[idx] = koff;
        c_klen[idx] = len;
        const uint4 *src = reinterpret_cast<const uint4 *>(t.arena + t.row_off[r]);
        uint4 *dst = reinterpret_cast<uint4 *>(c_keys + koff);
        for (uint32_t q = 0; q < padded / 16; ++q) dst[q] = src[q];
    }
}

int launch_partition_fill(const DevTable &t, uint64_t rows, uint32_t n_parts, uint32_t self, bool release,
                          uint8_t *buf, const uint64_t *d_chunk_off, const uint64_t *d_part_rows,
                          const uint64_t *d_part_keybytes, unsigned long long *cursors,
                          cudaStream_t st, uint32_t umi_len)
{
    uint64_t blocks = (rows + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    if (blocks < 1) blocks = 1;
    if (umi_len)
        k5_partition_fill<true><<<(uint32_t)blocks, 256, 0, st>>>(t, rows, n_parts, self, release, buf, d_chunk_off,
                                                                  d_part_rows, d_part_keybytes, cursors, umi_len);
    else
        k5_partition_fill<false><<<(uint32_t)blocks, 256, 0, st>>>(t, rows, n_parts, self, release, buf, d_chunk_off,
                                                                   d_part_rows, d_part_keybytes, cursors, 0);
    ++g_launches;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

}  // namespace vfb

extern "C" int vfb_debug_translate12(const uint8_t *bases12, uint8_t *aa4, int *canonical)
{
    if (!bases12 || !aa4 || !canonical) { vfb::set_error("null argument"); return VFB_ERR_ARG; }
    static const char aa64[65] =
        "KNKN" "TTTT" "RSRS" "IIMI"
        "QHQH" "PPPP" "RRRR" "LLLL"
        "EDED" "AAAA" "GGGG" "VVVV"
        "*Y*Y" "SSSS" "*CWC" "LFLF";
    uint32_t x[3];
    for (int k = 0; k < 3; ++k)
        x[k] = (uint32_t)bases12[4 * k] | ((uint32_t)bases12[4 * k + 1] << 8) | ((uint32_t)bases12[4 * k + 2] << 16) |
               ((uint32_t)bases12[4 * k + 3] << 24);
    uint32_t i[4];
    *canonical = tf_codons12(x[0], x[1], x[2], i[0], i[1], i[2], i[3]) ? 1 : 0;
    for (int k = 0; k < 4; ++k) aa4[k] = tf_codon_entry(i[k] & 0xFFFu, aa64);
    return VFB_OK;
}
