// umi_length: the count table holds (variant, UMI) rows, the key being the variant's bytes followed by umi_len UMI
// bytes.  At finish the export's count column is grouped by variant: every row with a count is inserted into an
// open-addressed slot table keyed by the multilinear hash of its variant part (debug_hash_bits keeps only its low bits);
// membership is decided on the variant bytes.  The first row to claim a slot represents the group and ends with the
// group's summed count and its number of rows (distinct UMIs = molecules); the other rows end with count 0, so the
// export's compaction drops them.  The count table itself is not touched.
// The claim-or-find loop is the one k_col_dups (kernels_collapse.cu) runs, with a variant-length compare; it is not
// shared because k_col_dups compiled through a shared helper is different machine code, and collapse_ratio's kernels are
// kept exactly as they were.
#include "ctx.cuh"
#include "hash.h"

namespace vfb {

namespace {

// word i of a key in the arena (16-byte aligned, zero-padded) with the bytes at or past len cleared
__device__ __forceinline__ uint32_t umi_word(const uint32_t *k, uint32_t len, uint32_t i)
{
    const uint32_t w = k[i], left = len - 4 * i;
    return left < 4 ? w & ((1u << (8 * left)) - 1u) : w;
}

// A slot is 16 bytes: [0] = rows of the group (molecules) << 32 | representative row + 1 (0 = empty; rows < 2^30), [1] the
// group's summed count.
__global__ void __launch_bounds__(256)
k_umi_group(const DevTable t, const unsigned long long *count, uint64_t rows, uint32_t umi_len, unsigned long long *slots,
            uint64_t mask, int hash_bits, uint32_t *slot_of)
{
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += stride) {
        const unsigned long long c = count[r];
        if (!c) continue;
        const uint32_t full = t.row_len[r], len = full - umi_len;
        const uint32_t *k = reinterpret_cast<const uint32_t *>(t.arena + t.row_off[r]);
        const uint32_t nw = (len + 3) / 4;
        uint64_t acc = 0;
        for (uint32_t i = 0; i < nw; ++i) acc += vfb_hash_term(umi_word(k, len, i), i);
        uint64_t h = vfb_hash_finish(acc, len);
        if (hash_bits > 0 && hash_bits < 64) h &= (1ull << hash_bits) - 1;
        const unsigned long long mine = 1ull << 32 | (r + 1);
        uint64_t s = h & mask;
        bool claimed = false;
        for (;; s = (s + 1) & mask) {
            unsigned long long cur = slots[2 * s];
            if (cur == 0ull) {
                cur = atomicCAS(&slots[2 * s], 0ull, mine);
                if (cur == 0ull) { claimed = true; break; }
            }
            const uint64_t q = (uint32_t)cur - 1;
            if (t.row_len[q] != full) continue;        // one umi_len for every row: equal lengths <=> equal variant lengths
            const uint32_t *kq = reinterpret_cast<const uint32_t *>(t.arena + t.row_off[q]);
            uint32_t diff = 0;
            for (uint32_t i = 0; i < nw; ++i) diff |= umi_word(k, len, i) ^ umi_word(kq, len, i);
            if (diff == 0u) break;
        }
        if (!claimed) atomicAdd(&slots[2 * s], 1ull << 32);
        atomicAdd(&slots[2 * s + 1], c);
        slot_of[r] = (uint32_t)s;
    }
}

// stats: [0] rows with a count (pairs), [1] groups (variant rows)
__global__ void __launch_bounds__(256)
k_umi_fold(uint64_t rows, unsigned long long *count, const unsigned long long *slots, const uint32_t *slot_of,
           unsigned long long *row_mol, unsigned long long *stats)
{
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    uint32_t pairs = 0, groups = 0;
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += stride) {
        if (!count[r]) continue;
        const uint64_t s = slot_of[r];
        ++pairs;
        const unsigned long long w = slots[2 * s];
        if ((uint32_t)w == r + 1) {
            count[r] = slots[2 * s + 1];
            row_mol[r] = w >> 32;
            ++groups;
        } else {
            count[r] = 0ull;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        pairs += __shfl_xor_sync(0xffffffffu, pairs, o);
        groups += __shfl_xor_sync(0xffffffffu, groups, o);
    }
    if ((threadIdx.x & 31) == 0 && pairs) {
        atomicAdd(&stats[0], (unsigned long long)pairs);
        atomicAdd(&stats[1], (unsigned long long)groups);
    }
}

uint32_t umi_grid(uint64_t items)
{
    uint64_t b = (items + 255) / 256;
    if (b > 148 * 16) b = 148 * 16;
    return (uint32_t)(b ? b : 1);
}

}  // namespace

int umi_group_rows(const DevTable &t, unsigned long long *count, unsigned long long *row_mol, uint64_t rows, uint32_t umi_len,
                   int hash_bits, cudaStream_t st, uint64_t *pairs, uint64_t *groups, float *ms)
{
    *pairs = *groups = 0;
    *ms = 0.f;
    if (rows == 0) return VFB_OK;
    // scratch: a table of 16-byte slots at most half full and a 4-byte slot index per row, 36-68 bytes per row (at most
    // 2^31 slots: 32 GiB at the limit); one pass, as a row's group must be found among all rows
    if (rows >= (1ull << 30)) { set_error("umi: 2^30 or more (variant, UMI) rows are not supported"); return VFB_ERR_ARG; }
    uint64_t cap = 1024;
    while (cap < 2 * rows) cap <<= 1;
    struct Scratch {
        cudaStream_t st;
        DevBuf slots, slot_of, stats;
        cudaEvent_t ev[2] = {nullptr, nullptr};
        ~Scratch()
        {
            cudaStreamSynchronize(st);
            slots.release(); slot_of.release(); stats.release();
            for (cudaEvent_t e : ev) if (e) cudaEventDestroy(e);
        }
    } x{st};
    int rc;
    VFB_CUDA(cudaEventCreate(&x.ev[0]));
    VFB_CUDA(cudaEventCreate(&x.ev[1]));
    if ((rc = x.slots.ensure(cap * 16)) || (rc = x.slot_of.ensure(rows * 4)) || (rc = x.stats.ensure(16))) return rc;
    VFB_CUDA(cudaEventRecord(x.ev[0], st));
    VFB_CUDA(cudaMemsetAsync(x.slots.p, 0, cap * 16, st));
    VFB_CUDA(cudaMemsetAsync(x.stats.p, 0, 16, st));
    unsigned long long *sl = x.slots.as<unsigned long long>();
    k_umi_group<<<umi_grid(rows), 256, 0, st>>>(t, count, rows, umi_len, sl, cap - 1, hash_bits, x.slot_of.as<uint32_t>());
    k_umi_fold<<<umi_grid(rows), 256, 0, st>>>(rows, count, sl, x.slot_of.as<uint32_t>(), row_mol, x.stats.as<unsigned long long>());
    g_launches += 2;
    VFB_CUDA(cudaGetLastError());
    VFB_CUDA(cudaEventRecord(x.ev[1], st));
    unsigned long long h[2];
    VFB_CUDA(cudaMemcpyAsync(h, x.stats.p, 16, cudaMemcpyDeviceToHost, st));
    VFB_CUDA(cudaStreamSynchronize(st));
    VFB_CUDA(cudaEventElapsedTime(ms, x.ev[0], x.ev[1]));
    *pairs = h[0];
    *groups = h[1];
    return VFB_OK;
}

}  // namespace vfb
