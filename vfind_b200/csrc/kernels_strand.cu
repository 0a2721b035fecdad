// both_strands: the reverse-complement gather between a batch's forward pass and its reverse pass.
//
// A read is retried on the reverse strand iff it is not empty and the forward pass left it without a region
// (start, end located, start < end <= len: the predicate of the key kernels).  k_strand_gather writes the reverse
// complement of every such read into a lane-owned text buffer, back to back, with a compact span list and the
// original index of each gathered read.  One 64-bit atomic per warp claims both the compact indices (high word) and
// the text range (low word), so compact order is text order: the 32 reads of a scan or key unit of the reverse pass
// are adjacent in memory and the tile kernels stage them with one bulk copy.
#include "vfb_internal.cuh"

namespace vfb {

// A <-> T, C <-> G (either case), U -> A, u -> a; every other byte stays as it is.
__host__ __device__ __forceinline__ uint8_t rc_base(uint8_t b)
{
    switch (b) {
    case 'A': return 'T';
    case 'T': return 'A';
    case 'U': return 'A';
    case 'C': return 'G';
    case 'G': return 'C';
    case 'a': return 't';
    case 't': return 'a';
    case 'u': return 'a';
    case 'c': return 'g';
    case 'g': return 'c';
    default: return b;
    }
}

#define STRAND_THREADS 256

// The warp writes the reverse complement of text[so, so+len) to out[d0, d0+len): one lane per aligned 16-byte chunk of
// the destination, a 16-byte store where the chunk lies inside the read, byte stores at the two ends (the chunks there
// are shared with the neighbouring reads, which other warps write).
__device__ __forceinline__ void rc_copy(const uint8_t *__restrict__ text, uint32_t so, uint32_t len, uint8_t *__restrict__ out,
                                        uint32_t d0, const uint8_t *lut, int lane)
{
    const uint64_t lo = d0, hi = (uint64_t)d0 + len;      // (64-bit: the gathered text may end at 2^32)
    const uint8_t *src_end = text + so + len - 1;          // destination byte d0 + t comes from src_end[-t]
    for (uint64_t c = (lo >> 4) + (uint64_t)lane; c <= (hi - 1) >> 4; c += 32) {
        const uint64_t p0 = c << 4;
        if (p0 >= lo && p0 + 16 <= hi) {
            const uint8_t *s = src_end - (p0 - d0);
            uint32_t w[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t b0 = lut[__ldg(s - 4 * k)], b1 = lut[__ldg(s - 4 * k - 1)];
                const uint32_t b2 = lut[__ldg(s - 4 * k - 2)], b3 = lut[__ldg(s - 4 * k - 3)];
                w[k] = b0 | (b1 << 8) | (b2 << 16) | (b3 << 24);
            }
            *reinterpret_cast<uint4 *>(out + p0) = make_uint4(w[0], w[1], w[2], w[3]);
        } else {
            for (uint64_t p = p0 < lo ? lo : p0; p < p0 + 16 && p < hi; ++p) out[p] = lut[__ldg(src_end - (p - lo))];
        }
    }
}

__global__ void __launch_bounds__(STRAND_THREADS)
k_strand_gather(const vfb_span *__restrict__ spans, const uint32_t *__restrict__ start, const uint32_t *__restrict__ end,
                uint32_t n, const uint8_t *__restrict__ text, uint8_t *__restrict__ out, vfb_span *__restrict__ out_spans,
                uint32_t *__restrict__ src, unsigned long long *cursor, unsigned long long *n_gathered)
{
    __shared__ uint8_t lut[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) lut[i] = rc_base((uint8_t)i);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const uint32_t warps_total = gridDim.x * (STRAND_THREADS / 32);
    const uint32_t n_units = (n + 31) / 32;
    for (uint32_t unit = blockIdx.x * (STRAND_THREADS / 32) + (threadIdx.x >> 5); unit < n_units; unit += warps_total) {
        const uint32_t r = unit * 32 + lane;
        bool need = false;
        vfb_span sp = vfb_span{0u, 0u};
        if (r < n) {
            sp = spans[r];
            const uint32_t s = start[r], e = end[r];
            const bool region = s != VFB_NONE && e != VFB_NONE && s < e && e <= sp.len;
            need = !region && sp.len > 0;
        }
        const unsigned mask = __ballot_sync(0xffffffffu, need);
        if (mask == 0) continue;
        const uint32_t len = need ? sp.len : 0u;
        uint32_t incl = len;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
        const uint32_t cnt = (uint32_t)__popc(mask);
        unsigned long long old = 0;
        if (lane == 0) {
            old = atomicAdd(cursor, ((unsigned long long)cnt << 32) | total);
            atomicAdd(n_gathered, (unsigned long long)cnt);
        }
        old = __shfl_sync(0xffffffffu, old, 0);
        const uint32_t d0 = (uint32_t)old + (incl - len);
        if (need) {
            const uint32_t idx = (uint32_t)(old >> 32) + (uint32_t)__popc(mask & ((1u << lane) - 1u));
            out_spans[idx] = vfb_span{d0, len};
            src[idx] = r;
        }
        unsigned todo = mask;
        while (todo) {
            const int q = __ffs((int)todo) - 1;
            todo &= todo - 1;
            rc_copy(text, __shfl_sync(0xffffffffu, sp.off, q), __shfl_sync(0xffffffffu, len, q), out,
                    __shfl_sync(0xffffffffu, d0, q), lut, lane);
        }
    }
}

// t64[0] -= counted (before the reverse keys) or += counted (after the reverse inserts): the reads counted in between.
__global__ void k_strand_tally(unsigned long long *t64, const unsigned long long *counters, int after)
{
    if (after) *t64 += counters[2];
    else *t64 -= counters[2];
}

int launch_strand_gather(const StrandJob &j, int sm_count, cudaStream_t st)
{
    if (j.n == 0) return VFB_OK;
    uint32_t blocks = (j.n + STRAND_THREADS - 1) / STRAND_THREADS;
    const uint32_t cap = (uint32_t)sm_count * 8u;
    if (blocks > cap) blocks = cap;
    k_strand_gather<<<blocks, STRAND_THREADS, 0, st>>>(j.spans, j.start, j.end, j.n, j.text, j.out, j.out_spans, j.src,
                                                       j.cursor, j.n_gathered);
    ++g_launches;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

int launch_strand_tally(unsigned long long *t64, const unsigned long long *counters, bool after, cudaStream_t st)
{
    k_strand_tally<<<1, 1, 0, st>>>(t64, counters, after ? 1 : 0);
    ++g_launches;
    VFB_CUDA(cudaGetLastError());
    return VFB_OK;
}

}  // namespace vfb

extern "C" int vfb_debug_revcomp(const uint8_t *in, uint64_t n, uint8_t *out)
{
    if (n && (!in || !out)) { vfb::set_error("null argument"); return VFB_ERR_ARG; }
    for (uint64_t i = 0; i < n; ++i) out[i] = vfb::rc_base(in[n - 1 - i]);
    return VFB_OK;
}
