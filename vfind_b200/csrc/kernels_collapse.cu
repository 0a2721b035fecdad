// collapse_ratio: fold every row into a more abundant neighbour one byte substitution away (directional clustering).
//
// Order: count descending, then key bytes ascending.  a may be the parent of b when they have the same length and
// differ in exactly one byte, a comes first in the order and (double)count(a) >= ratio * (double)count(b); parent(b)
// is the first such a.  Every row's count goes to the end of its parent chain (its root).
//
// Scheme (masked-position grouping): the keys that agree everywhere except at position p form one group of (len, p).
// Every (row, p) pair is inserted once into an open-addressed group table, a range of positions per pass.  Inside a
// group all members differ only at p, so the group's first member in the order is the atomicMax of
// count << 8 | (255 - key[p]) (counts < 2^56).  A row's candidate at p is that member, unless it is the row itself;
// if it fails the ratio every other member fails it too.  Candidates of one row at different positions are ordered
// without key bytes of the candidates: at equal counts, the candidate differing from row r at the smaller position q
// with byte x comes first iff x < r[q].  Roots are found by pointer jumping, then children add into their roots.
//
// The group table places a pair by the masked multilinear hash of hash.h (the row's accumulator with one word's term
// replaced, O(1) per position); membership is decided on position, length and the full key bytes, so the result does
// not depend on the hash (debug_hash_bits keeps only its low bits).
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <vector>

#include "ctx.cuh"
#include "hash.h"

namespace vfb {

namespace {

// flags word bits
enum { CF_DUPLICATE = 1u, CF_BIG_COUNT = 2u, CF_LONG_KEY = 4u };

struct Rows {
    const uint8_t *keys;
    const uint64_t *off;
    const uint32_t *len;
    unsigned long long *count;
    uint64_t n;
};

__device__ __forceinline__ uint32_t load_word(const uint8_t *k, uint32_t len, uint32_t i)
{
    uint32_t w = 0;
#pragma unroll
    for (uint32_t b = 0; b < 4; ++b) {
        const uint32_t q = i * 4 + b;
        if (q < len) w |= (uint32_t)k[q] << (8 * b);
    }
    return w;
}

// masked hash of (row, p): the accumulator with word p/4's term replaced by the term of that word with byte p cleared
__device__ __forceinline__ uint64_t masked_acc(uint64_t acc, uint32_t w, uint32_t p)
{
    const uint32_t i = p >> 2;
    const uint32_t wm = w & ~(0xFFu << (8 * (p & 3u)));
    return acc - vfb_hash_term(w, i) + vfb_hash_term(wm, i);
}

__device__ __forceinline__ uint64_t pair_hash(uint64_t macc, uint32_t len, uint32_t p, int hash_bits)
{
    uint64_t h = vfb_fmix64(vfb_hash_finish(macc, len) ^ ((uint64_t)(p + 1) * 0x9E3779B97F4A7C15ull));
    if (hash_bits > 0 && hash_bits < 64) h &= (1ull << hash_bits) - 1;
    return h;
}

__global__ void __launch_bounds__(256)
k_col_prep(Rows v, uint64_t *acc, uint32_t *cand_row, unsigned long long *stats /* [0] rows in, [1] max len */,
           unsigned int *flags)
{
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < v.n; r += stride) {
        cand_row[r] = VFB_NONE;
        const unsigned long long c = v.count[r];
        if (!c) continue;
        if (c >> 56) atomicOr(flags, (unsigned)CF_BIG_COUNT);
        const uint32_t len = v.len[r];
        if (len >= (1u << 24)) atomicOr(flags, (unsigned)CF_LONG_KEY);
        const uint8_t *k = v.keys + v.off[r];
        uint64_t a = 0;
        for (uint32_t i = 0; i < (len + 3) / 4; ++i) a += vfb_hash_term(load_word(k, len, i), i);
        acc[r] = a;
        atomicAdd(&stats[0], 1ull);
        atomicMax(&stats[1], (unsigned long long)len);
    }
}

// Whole keys into the slot table (position field VFB_NONE), before any masked pass: two rows with the same bytes are a
// duplicate.  Every row with a count is inserted, and equality is decided on the full bytes, so a duplicate is found
// whichever row claims the slot.
__global__ void __launch_bounds__(256)
k_col_dups(Rows v, const uint64_t *acc, unsigned long long *slots, uint64_t mask, int hash_bits, unsigned int *flags)
{
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < v.n; r += stride) {
        if (!v.count[r]) continue;
        const uint32_t len = v.len[r];
        const uint8_t *k = v.keys + v.off[r];
        const unsigned long long mine = (unsigned long long)VFB_NONE << 32 | (r + 1);
        for (uint64_t s = pair_hash(acc[r], len, VFB_NONE, hash_bits) & mask;; s = (s + 1) & mask) {
            unsigned long long cur = slots[2 * s];
            if (cur == 0ull) {
                cur = atomicCAS(&slots[2 * s], 0ull, mine);
                if (cur == 0ull) break;
            }
            const uint64_t q = (cur & 0xFFFFFFFFull) - 1;
            if (v.len[q] != len || acc[q] != acc[r]) continue;
            const uint8_t *kq = v.keys + v.off[q];
            bool same = true;
            for (uint32_t b = 0; b < len && same; ++b) same = k[b] == kq[b];
            if (same) { atomicOr(flags, (unsigned)CF_DUPLICATE); break; }
        }
    }
}

// A slot is two words: [0] = p << 32 | (representative row + 1) (0 = empty), [1] = the group's best (atomicMax).
// After k_col_best_row, word [0] holds p << 32 | (best row + 1).
__global__ void __launch_bounds__(256)
k_col_insert(Rows v, const uint64_t *acc, uint32_t p0, uint32_t np, unsigned long long *slots, uint64_t mask,
             uint32_t *slot_of, int hash_bits)
{
    const uint64_t pairs = v.n * np;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < pairs; j += stride) {
        const uint64_t r = j / np;
        const uint32_t p = p0 + (uint32_t)(j - r * np);
        const uint32_t len = v.len[r];
        if (p >= len || !v.count[r]) { slot_of[j] = VFB_NONE; continue; }
        const uint8_t *k = v.keys + v.off[r];
        const uint32_t w = load_word(k, len, p >> 2);
        const uint64_t macc = masked_acc(acc[r], w, p);
        const unsigned long long mine = (unsigned long long)p << 32 | (r + 1);
        uint64_t s = pair_hash(macc, len, p, hash_bits) & mask;
        for (;;) {
            unsigned long long cur = slots[2 * s];
            if (cur == 0ull) {
                cur = atomicCAS(&slots[2 * s], 0ull, mine);
                if (cur == 0ull) break;
            }
            if ((uint32_t)(cur >> 32) == p) {
                const uint64_t q = (cur & 0xFFFFFFFFull) - 1;
                if (v.len[q] == len) {
                    const uint8_t *kq = v.keys + v.off[q];
                    if (masked_acc(acc[q], load_word(kq, len, p >> 2), p) == macc) {
                        bool same = true;
                        for (uint32_t b = 0; b < len && same; ++b) same = b == p || k[b] == kq[b];
                        if (same) break;
                    }
                }
            }
            s = (s + 1) & mask;
        }
        slot_of[j] = (uint32_t)s;
    }
}

__device__ __forceinline__ unsigned long long best_word(unsigned long long count, uint8_t x)
{
    return count << 8 | (unsigned long long)(255u - x);
}

__global__ void __launch_bounds__(256)
k_col_best(Rows v, uint32_t p0, uint32_t np, unsigned long long *slots, const uint32_t *slot_of)
{
    const uint64_t pairs = v.n * np;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < pairs; j += stride) {
        const uint32_t s = slot_of[j];
        if (s == VFB_NONE) continue;
        const uint64_t r = j / np;
        const uint32_t p = p0 + (uint32_t)(j - r * np);
        atomicMax(&slots[2 * (uint64_t)s + 1], best_word(v.count[r], v.keys[v.off[r] + p]));
    }
}

__global__ void __launch_bounds__(256)
k_col_best_row(Rows v, uint32_t p0, uint32_t np, unsigned long long *slots, const uint32_t *slot_of)
{
    const uint64_t pairs = v.n * np;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < pairs; j += stride) {
        const uint32_t s = slot_of[j];
        if (s == VFB_NONE) continue;
        const uint64_t r = j / np;
        const uint32_t p = p0 + (uint32_t)(j - r * np);
        // exactly one member matches: the others differ from it at p (k_col_dups has ruled out duplicate keys)
        if (slots[2 * (uint64_t)s + 1] == best_word(v.count[r], v.keys[v.off[r] + p]))
            slots[2 * (uint64_t)s] = (unsigned long long)p << 32 | (r + 1);
    }
}

// One thread per row over the positions of the pass: the row's candidate parent so far is (cand_row, count of it,
// cand_px = p << 8 | its byte at p).
__global__ void __launch_bounds__(256)
k_col_candidate(Rows v, uint32_t p0, uint32_t np, const unsigned long long *slots, const uint32_t *slot_of, double ratio,
                uint32_t *cand_row, unsigned long long *cand_cnt, uint32_t *cand_px)
{
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < v.n; r += stride) {
        const unsigned long long c = v.count[r];
        const uint32_t len = v.len[r];
        if (!c || len <= p0) continue;
        const uint8_t *k = v.keys + v.off[r];
        const double need = __dmul_rn(ratio, __ull2double_rn(c));
        uint32_t row = cand_row[r], px = 0;
        unsigned long long cc = 0;
        if (row != VFB_NONE) { cc = cand_cnt[r]; px = cand_px[r]; }
        const uint32_t pe = min(p0 + np, len);
        for (uint32_t p = p0; p < pe; ++p) {
            const uint32_t s = slot_of[r * np + (p - p0)];
            const unsigned long long w0 = slots[2 * (uint64_t)s], w1 = slots[2 * (uint64_t)s + 1];
            const uint32_t best = (uint32_t)(w0 & 0xFFFFFFFFull) - 1;
            if (best == (uint32_t)r) continue;
            const unsigned long long bc = w1 >> 8;
            if (!(__ull2double_rn(bc) >= need)) continue;
            const uint32_t x = 255u - (uint32_t)(w1 & 0xFFu);
            bool take;
            if (row == VFB_NONE || bc > cc) take = true;
            else if (bc < cc) take = false;
            else {
                const uint32_t cp = px >> 8, cx = px & 0xFFu;
                if (p == cp) take = x < cx;
                else if (p < cp) take = x < k[p];        // differs from r first at p: earlier iff its byte is smaller
                else take = !(cx < k[cp]);               // the current one differs first at cp
            }
            if (take) { row = best; cc = bc; px = p << 8 | x; }
        }
        if (row != VFB_NONE) { cand_row[r] = row; cand_cnt[r] = cc; cand_px[r] = px; }
    }
}

__global__ void __launch_bounds__(256)
k_col_parent(uint64_t n, const uint32_t *cand_row, uint32_t *parent)
{
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += stride)
        parent[r] = cand_row[r] == VFB_NONE ? (uint32_t)r : cand_row[r];
}

__global__ void __launch_bounds__(256)
k_col_jump(uint64_t n, uint32_t *parent, unsigned int *changed)
{
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    bool any = false;
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += stride) {
        const uint32_t a = parent[r], b = parent[a];
        if (a != b) { parent[r] = b; any = true; }
    }
    if (any) *changed = 1u;
}

__global__ void __launch_bounds__(256)
k_col_fold(Rows v, const uint32_t *parent, unsigned long long *stats /* [2] roots */)
{
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < v.n; r += stride) {
        const unsigned long long c = v.count[r];
        if (!c) continue;
        const uint32_t root = parent[r];
        if (root == (uint32_t)r) { atomicAdd(&stats[2], 1ull); continue; }
        atomicAdd(&v.count[root], c);
        v.count[r] = 0ull;
    }
}

uint32_t grid_for(uint64_t items)
{
    uint64_t b = (items + 255) / 256;
    if (b > 148 * 16) b = 148 * 16;
    return (uint32_t)(b ? b : 1);
}

uint64_t pow2_ge(uint64_t v)
{
    uint64_t p = 1024;
    while (p < v) p <<= 1;
    return p;
}

}  // namespace

int collapse_rows(const uint8_t *keys, const uint64_t *off, const uint32_t *len, unsigned long long *count, uint64_t rows,
                  double ratio, int hash_bits, cudaStream_t st, uint64_t *rows_in, uint64_t *rows_out, float *ms)
{
    *rows_in = *rows_out = 0;
    *ms = 0.f;
    if (rows == 0) return VFB_OK;
    // a pass holds every row at one position at least: 2^29 rows fill a table of 2^30 slots, whose indices slot_of holds
    if (rows > VFB_COLLAPSE_MAX_ROWS) { set_error("collapse: more than 2^29 rows are not supported"); return VFB_ERR_ARG; }
    const Rows v{keys, off, len, count, rows};
    // scratch goes back to the device pool when the call returns, after the stream has drained
    struct Scratch {
        cudaStream_t st;
        DevBuf acc, cand_row, cand_cnt, cand_px, parent, small, slots, slot_of;
        cudaEvent_t ev[2] = {nullptr, nullptr};
        ~Scratch()
        {
            cudaStreamSynchronize(st);
            for (DevBuf *b : {&acc, &cand_row, &cand_cnt, &cand_px, &parent, &small, &slots, &slot_of}) b->release();
            for (cudaEvent_t e : ev) if (e) cudaEventDestroy(e);
        }
    } x{st};
    int rc;
    VFB_CUDA(cudaEventCreate(&x.ev[0]));
    VFB_CUDA(cudaEventCreate(&x.ev[1]));
    if ((rc = x.acc.ensure(rows * 8)) || (rc = x.cand_row.ensure(rows * 4)) || (rc = x.cand_cnt.ensure(rows * 8)) ||
        (rc = x.cand_px.ensure(rows * 4)) || (rc = x.parent.ensure(rows * 4)) || (rc = x.small.ensure(64)))
        return rc;
    unsigned long long *stats = x.small.as<unsigned long long>();          // [0] rows in, [1] max len, [2] roots
    unsigned int *flags = reinterpret_cast<unsigned int *>(stats + 4), *changed = flags + 1;
    VFB_CUDA(cudaEventRecord(x.ev[0], st));
    VFB_CUDA(cudaMemsetAsync(x.small.p, 0, 64, st));
    k_col_prep<<<grid_for(rows), 256, 0, st>>>(v, x.acc.as<uint64_t>(), x.cand_row.as<uint32_t>(), stats, flags);
    ++g_launches;
    VFB_CUDA(cudaGetLastError());
    unsigned long long h[5];
    VFB_CUDA(cudaMemcpyAsync(h, x.small.p, 40, cudaMemcpyDeviceToHost, st));
    VFB_CUDA(cudaStreamSynchronize(st));
    const uint32_t hflags = (uint32_t)h[4];
    if (hflags & CF_BIG_COUNT) { set_error("collapse: counts must be below 2^56"); return VFB_ERR_VALUE; }
    if (hflags & CF_LONG_KEY) { set_error("collapse: keys must be shorter than 2^24 bytes"); return VFB_ERR_VALUE; }
    *rows_in = h[0];
    const uint32_t max_len = (uint32_t)h[1];
    {
        const uint64_t cap = pow2_ge(2 * rows);
        unsigned int fl = 0;
        if ((rc = x.slots.ensure(cap * 16))) return rc;
        VFB_CUDA(cudaMemsetAsync(x.slots.p, 0, cap * 16, st));
        k_col_dups<<<grid_for(rows), 256, 0, st>>>(v, x.acc.as<uint64_t>(), x.slots.as<unsigned long long>(), cap - 1,
                                                   hash_bits, flags);
        ++g_launches;
        VFB_CUDA(cudaGetLastError());
        VFB_CUDA(cudaMemcpyAsync(&fl, flags, 4, cudaMemcpyDeviceToHost, st));
        VFB_CUDA(cudaStreamSynchronize(st));
        if (fl & CF_DUPLICATE) { set_error("collapse: the table holds the same key twice"); return VFB_ERR_VALUE; }
    }

    // positions per pass: a pair costs a slot index (4 bytes) and up to two slots of 16 bytes at most half full
    size_t free_b = 0, total_b = 0;
    VFB_CUDA(cudaMemGetInfo(&free_b, &total_b));
    const uint64_t budget = std::max<uint64_t>((uint64_t)(free_b / 2), 256ull << 20);
    uint64_t max_pairs = budget / 68;
    max_pairs = std::min<uint64_t>(std::max<uint64_t>(max_pairs, rows), VFB_COLLAPSE_MAX_ROWS);
    uint32_t np = (uint32_t)std::min<uint64_t>(max_len, std::max<uint64_t>(1, max_pairs / rows));
    for (uint32_t p0 = 0; p0 < max_len; p0 += np) {
        const uint32_t n_here = std::min<uint32_t>(np, max_len - p0);
        const uint64_t pairs = rows * n_here;
        const uint64_t cap = pow2_ge(2 * pairs);
        if ((rc = x.slots.ensure(cap * 16)) || (rc = x.slot_of.ensure(pairs * 4))) return rc;
        VFB_CUDA(cudaMemsetAsync(x.slots.p, 0, cap * 16, st));
        unsigned long long *sl = x.slots.as<unsigned long long>();
        uint32_t *so = x.slot_of.as<uint32_t>();
        k_col_insert<<<grid_for(pairs), 256, 0, st>>>(v, x.acc.as<uint64_t>(), p0, n_here, sl, cap - 1, so, hash_bits);
        k_col_best<<<grid_for(pairs), 256, 0, st>>>(v, p0, n_here, sl, so);
        k_col_best_row<<<grid_for(pairs), 256, 0, st>>>(v, p0, n_here, sl, so);
        k_col_candidate<<<grid_for(rows), 256, 0, st>>>(v, p0, n_here, sl, so, ratio, x.cand_row.as<uint32_t>(),
                                                        x.cand_cnt.as<unsigned long long>(), x.cand_px.as<uint32_t>());
        g_launches += 4;
        VFB_CUDA(cudaGetLastError());
    }
    uint32_t *par = x.parent.as<uint32_t>();
    k_col_parent<<<grid_for(rows), 256, 0, st>>>(rows, x.cand_row.as<uint32_t>(), par);
    ++g_launches;
    VFB_CUDA(cudaGetLastError());
    // pointer jumping: the longest chain halves per launch
    for (;;) {
        unsigned int ch = 0;
        VFB_CUDA(cudaMemsetAsync(changed, 0, 4, st));
        k_col_jump<<<grid_for(rows), 256, 0, st>>>(rows, par, changed);
        ++g_launches;
        VFB_CUDA(cudaGetLastError());
        VFB_CUDA(cudaMemcpyAsync(&ch, changed, 4, cudaMemcpyDeviceToHost, st));
        VFB_CUDA(cudaStreamSynchronize(st));
        if (!ch) break;
    }
    k_col_fold<<<grid_for(rows), 256, 0, st>>>(v, par, stats);
    ++g_launches;
    VFB_CUDA(cudaGetLastError());
    VFB_CUDA(cudaEventRecord(x.ev[1], st));
    VFB_CUDA(cudaMemcpyAsync(h, stats, 24, cudaMemcpyDeviceToHost, st));
    VFB_CUDA(cudaStreamSynchronize(st));
    VFB_CUDA(cudaEventElapsedTime(ms, x.ev[0], x.ev[1]));
    *rows_out = h[2];
    return VFB_OK;
}

bool collapse_ratio_ok(double ratio) { return std::isfinite(ratio) && ratio >= 1.0; }

// Host columns -> device -> collapse -> the export's compaction -> host columns that `alloc` provides for the result's
// size (they may be the input's own buffers: the input has been uploaded by then, and the result is never larger).
int collapse_columns(const vfb_table &in, double ratio, int device, int hash_bits,
                     const std::function<int(uint64_t rows, uint64_t bytes, vfb_table *out)> &alloc, vfb_table *out,
                     vfb_collapse_info *info)
{
    const uint64_t rows = in.rows;
    if (rows && (!in.offsets || !in.counts)) { set_error("null column"); return VFB_ERR_ARG; }
    const uint64_t end = rows ? in.offsets[rows] : 0;
    if (end && !in.data) { set_error("null column"); return VFB_ERR_ARG; }
    if (end > in.key_bytes) { set_error("collapse: offsets past the end of the key bytes"); return VFB_ERR_ARG; }
    std::vector<uint32_t> len(rows);
    for (uint64_t r = 0; r < rows; ++r) {
        if (in.offsets[r] > in.offsets[r + 1]) { set_error("collapse: offsets must not decrease"); return VFB_ERR_ARG; }
        const uint64_t n = in.offsets[r + 1] - in.offsets[r];
        if (n >= (1u << 24)) { set_error("collapse: keys must be shorter than 2^24 bytes"); return VFB_ERR_VALUE; }
        len[r] = (uint32_t)n;
    }
    int prev = -1;
    VFB_CUDA(cudaGetDevice(&prev));
    if (device >= 0) VFB_CUDA(cudaSetDevice(device));
    struct Scope {
        int prev;
        cudaStream_t st = nullptr;
        DevBuf data, off, len, cnt, bbytes, brows, xoff, xcnt, xdata;
        ~Scope()
        {
            if (st) { cudaStreamSynchronize(st); cudaStreamDestroy(st); }
            for (DevBuf *b : {&data, &off, &len, &cnt, &bbytes, &brows, &xoff, &xcnt, &xdata}) b->release();
            cudaSetDevice(prev);
        }
    } x{prev};
    VFB_CUDA(cudaStreamCreateWithFlags(&x.st, cudaStreamNonBlocking));
    int rc;
    const uint64_t nb = (rows + 1023) / 1024;
    if ((rc = x.data.ensure(end ? end : 16)) || (rc = x.off.ensure(rows * 8 + 8)) || (rc = x.len.ensure(rows * 4 + 4)) ||
        (rc = x.cnt.ensure(rows * 8 + 8)) || (rc = x.bbytes.ensure((nb + 2) * 8)) || (rc = x.brows.ensure(nb * 8 + 8)))
        return rc;
    if (end) VFB_CUDA(cudaMemcpyAsync(x.data.p, in.data, end, cudaMemcpyHostToDevice, x.st));
    if (rows) {
        VFB_CUDA(cudaMemcpyAsync(x.off.p, in.offsets, rows * 8, cudaMemcpyHostToDevice, x.st));
        VFB_CUDA(cudaMemcpyAsync(x.len.p, len.data(), rows * 4, cudaMemcpyHostToDevice, x.st));
        VFB_CUDA(cudaMemcpyAsync(x.cnt.p, in.counts, rows * 8, cudaMemcpyHostToDevice, x.st));
    }
    uint64_t rows_in = 0, rows_out = 0;
    float ms = 0.f;
    if ((rc = collapse_rows(x.data.as<uint8_t>(), x.off.as<uint64_t>(), x.len.as<uint32_t>(), x.cnt.as<unsigned long long>(),
                            rows, ratio, hash_bits, x.st, &rows_in, &rows_out, &ms)))
        return rc;
    DevTable t{};
    t.arena = x.data.as<uint8_t>();
    t.row_off = x.off.as<uint64_t>();
    t.row_len = x.len.as<uint32_t>();
    unsigned long long *d_totals = x.bbytes.as<unsigned long long>() + nb, totals[2] = {0, 0};
    if ((rc = launch_export_sizes(t, rows, x.cnt.as<unsigned long long>(), x.bbytes.as<unsigned long long>(),
                                  x.brows.as<unsigned long long>(), d_totals, x.st)))
        return rc;
    if (rows) VFB_CUDA(cudaMemcpyAsync(totals, d_totals, 16, cudaMemcpyDeviceToHost, x.st));
    VFB_CUDA(cudaStreamSynchronize(x.st));
    const uint64_t out_bytes = totals[0], out_rows = totals[1];
    memset(out, 0, sizeof *out);
    if ((rc = alloc(out_rows, out_bytes, out))) return rc;
    out->rows = out_rows;
    out->key_bytes = out_bytes;
    if (out_rows) {
        if ((rc = x.xoff.ensure(out_rows * 8)) || (rc = x.xcnt.ensure(out_rows * 8)) || (rc = x.xdata.ensure(out_bytes ? out_bytes : 16)))
            return rc;
        if ((rc = launch_export_gather(t, rows, x.cnt.as<unsigned long long>(), x.bbytes.as<unsigned long long>(),
                                       x.brows.as<unsigned long long>(), 0, x.xoff.as<unsigned long long>(),
                                       x.xcnt.as<unsigned long long>(), x.xdata.as<uint8_t>(), x.st)))
            return rc;
        VFB_CUDA(cudaMemcpyAsync(out->offsets, x.xoff.p, out_rows * 8, cudaMemcpyDeviceToHost, x.st));
        VFB_CUDA(cudaMemcpyAsync(out->counts, x.xcnt.p, out_rows * 8, cudaMemcpyDeviceToHost, x.st));
        if (out_bytes) VFB_CUDA(cudaMemcpyAsync(out->data, x.xdata.p, out_bytes, cudaMemcpyDeviceToHost, x.st));
        VFB_CUDA(cudaStreamSynchronize(x.st));
    }
    out->offsets[out_rows] = out_bytes;
    if (info) { info->rows_in = rows_in; info->rows_out = rows_out; info->ms = ms; }
    return VFB_OK;
}

}  // namespace vfb

extern "C" int vfb_collapse(const vfb_table *in, double ratio, int device, int debug_hash_bits, vfb_table *out,
                            vfb_collapse_info *info)
{
    using namespace vfb;
    if (!in || !out) { set_error("null argument"); return VFB_ERR_ARG; }
    if (!collapse_ratio_ok(ratio)) { set_error("collapse ratio must be a finite number >= 1"); return VFB_ERR_VALUE; }
    memset(out, 0, sizeof *out);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        set_error("no CUDA device available (this library has no CPU fallback)");
        return VFB_ERR_CUDA;
    }
    auto alloc = [](uint64_t rows, uint64_t bytes, vfb_table *t) {
        t->offsets = (uint64_t *)malloc((rows + 1) * 8);
        t->counts = (uint64_t *)malloc(rows ? rows * 8 : 8);
        t->data = (uint8_t *)malloc(bytes ? bytes : 1);
        if (!t->offsets || !t->counts || !t->data) {
            free(t->offsets); free(t->counts); free(t->data);
            t->offsets = nullptr; t->counts = nullptr; t->data = nullptr;
            set_error("out of host memory");
            return (int)VFB_ERR_NOMEM;
        }
        return (int)VFB_OK;
    };
    const int rc = collapse_columns(*in, ratio, device, debug_hash_bits, alloc, out, info);
    if (rc) vfb_table_free(out);
    return rc;
}
