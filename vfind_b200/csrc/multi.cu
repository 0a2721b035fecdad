// Several devices behind one call (SURVEY §8(e)); the reference has no equivalent.
//
// vfb_multi_*: ONE process drives n devices — what `find_variants(path, ..., devices=[...])` and a Rust host that
// binds the C ABI use.  Reads shard across the devices with no data-path collective (ingest.cu deals block-gzip
// segments / inflated chunks round robin); the only exchange is the final merge of the per-device tables.
//
// The merge keeps every key on the device that owns it (owner = f(hash(key))): a device exports only the rows other
// devices own, one chunk per owner, and hands those rows' counts over; chunks travel
//   * by peer copies over NVLink (cudaMemcpyPeerAsync) when the devices share the process (vfb_multi_merge), or
//   * through NCCL send/recv (vfb_merge_nccl) when there is one process per device (torchrun, MPI): libnccl.so.2 is
//     loaded at run time (the library does not link it), the communicator is created from a 128-byte id that the
//     caller's own control plane carries from rank 0 to the others (vfb_nccl_unique_id / vfb_nccl_comm_init);
// and each device adds what it received with the same insert kernel that counts reads.  Counts are integers, so the
// merged table is bit-identical for any device count and any order of arrival.
#include <dlfcn.h>

#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "ctx.cuh"

using namespace vfb;

// ------------------------------------------------------------------------------------ NCCL at run time
namespace {

typedef struct { char internal[128]; } nccl_unique_id;
typedef void *nccl_comm;
enum { NCCL_UINT8 = 1, NCCL_UINT64 = 5 };

struct NcclApi {
    void *lib = nullptr;
    int (*GetUniqueId)(nccl_unique_id *) = nullptr;
    int (*CommInitRank)(nccl_comm *, int, nccl_unique_id, int) = nullptr;
    int (*CommDestroy)(nccl_comm) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, nccl_comm, cudaStream_t) = nullptr;
    int (*Send)(const void *, size_t, int, int, nccl_comm, cudaStream_t) = nullptr;
    int (*Recv)(void *, size_t, int, int, nccl_comm, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    std::string why;
};

NcclApi *nccl_api()
{
    static NcclApi *api = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        NcclApi *a = new NcclApi;
        const char *names[] = {getenv("VFB_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
        for (const char *n : names) {
            if (!n || !*n) continue;
            a->lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (a->lib) break;
            a->why = dlerror();
        }
        if (a->lib) {
            bool ok = true;
            auto sym = [&](const char *n) { void *p = dlsym(a->lib, n); if (!p) { ok = false; a->why = std::string("missing symbol ") + n; } return p; };
            a->GetUniqueId = (decltype(a->GetUniqueId))sym("ncclGetUniqueId");
            a->CommInitRank = (decltype(a->CommInitRank))sym("ncclCommInitRank");
            a->CommDestroy = (decltype(a->CommDestroy))sym("ncclCommDestroy");
            a->AllGather = (decltype(a->AllGather))sym("ncclAllGather");
            a->Send = (decltype(a->Send))sym("ncclSend");
            a->Recv = (decltype(a->Recv))sym("ncclRecv");
            a->GroupStart = (decltype(a->GroupStart))sym("ncclGroupStart");
            a->GroupEnd = (decltype(a->GroupEnd))sym("ncclGroupEnd");
            a->GetErrorString = (decltype(a->GetErrorString))sym("ncclGetErrorString");
            if (!ok) { dlclose(a->lib); a->lib = nullptr; }
        }
        api = a;
    });
    return api;
}

int nccl_need(NcclApi **out)
{
    NcclApi *a = nccl_api();
    if (!a->lib) {
        set_error("NCCL is not available (libnccl.so.2 could not be loaded; VFB_NCCL_LIB names it): " + a->why);
        return VFB_ERR_CUDA;
    }
    *out = a;
    return VFB_OK;
}

#define VFB_NCCL(a, call)                                                                   \
    do {                                                                                    \
        const int r__ = (call);                                                             \
        if (r__ != 0) {                                                                     \
            set_error(std::string("NCCL error: ") + (a)->GetErrorString(r__) + " in " #call); \
            return VFB_ERR_CUDA;                                                            \
        }                                                                                   \
    } while (0)

}  // namespace

extern "C" {

int vfb_nccl_available(void) { return nccl_api()->lib ? 1 : 0; }

int vfb_nccl_unique_id(uint8_t *id128)
{
    if (!id128) { set_error("null argument"); return VFB_ERR_ARG; }
    NcclApi *a;
    int rc = nccl_need(&a);
    if (rc) return rc;
    nccl_unique_id id;
    VFB_NCCL(a, a->GetUniqueId(&id));
    memcpy(id128, id.internal, 128);
    return VFB_OK;
}

int vfb_nccl_comm_init(const uint8_t *id128, uint32_t n_ranks, uint32_t rank, int device, void **comm_out)
{
    if (!id128 || !comm_out || n_ranks == 0 || rank >= n_ranks) { set_error("bad argument"); return VFB_ERR_ARG; }
    NcclApi *a;
    int rc = nccl_need(&a);
    if (rc) return rc;
    if (device >= 0) VFB_CUDA(cudaSetDevice(device));
    nccl_unique_id id;
    memcpy(id.internal, id128, 128);
    nccl_comm comm = nullptr;
    VFB_NCCL(a, a->CommInitRank(&comm, (int)n_ranks, id, (int)rank));
    *comm_out = comm;
    return VFB_OK;
}

int vfb_nccl_comm_destroy(void *comm)
{
    if (!comm) return VFB_OK;
    NcclApi *a;
    int rc = nccl_need(&a);
    if (rc) return rc;
    VFB_NCCL(a, a->CommDestroy((nccl_comm)comm));
    return VFB_OK;
}

// One process per device: afterwards this rank's table holds exactly the keys it owns, with global counts.
// Everything is queued on the context's compute stream; one host synchronisation (the part sizes of all ranks,
// gathered with one ncclAllGather straight from the counting kernel's output).
int vfb_merge_nccl(vfb_ctx *c, void *comm, uint32_t rank, uint32_t n_ranks)
{
    if (!c || !comm || n_ranks == 0 || rank >= n_ranks || n_ranks > 1024) { set_error("bad argument"); return VFB_ERR_ARG; }
    if (n_ranks == 1) return VFB_OK;
    NcclApi *a;
    int rc = nccl_need(&a);
    if (rc) return rc;
    const uint32_t n = n_ranks;
    const bool tr = trace_on();          // VFB_TRACE: synchronise between the phases and print their times
    auto stamp = [&](const char *what) {
        if (!tr) return;
        cudaStreamSynchronize(c->st_compute);
        trace("merge_nccl rank %u: %s", rank, what);
    };
    stamp("start (lanes joined)");
    if ((rc = vfb_internal_partition_count(c, n, rank, nullptr))) return rc;
    stamp("partition count");
    // every rank's [rows per part | key bytes per part]
    if ((rc = c->m_cursors.ensure((size_t)n * n * 16 + (size_t)n * 16))) return rc;     // gathered sizes live behind the cursors
    unsigned long long *d_all = c->m_cursors.as<unsigned long long>() + 2 * n;
    VFB_NCCL(a, a->AllGather(c->m_part_rows.p, d_all, (size_t)n * 2, NCCL_UINT64, (nccl_comm)comm, c->st_compute));
    std::vector<uint64_t> all((size_t)n * n * 2);
    VFB_CUDA(cudaMemcpyAsync(all.data(), d_all, all.size() * 8, cudaMemcpyDeviceToHost, c->st_compute));
    VFB_CUDA(cudaStreamSynchronize(c->st_compute));
    c->stats.d2h_bytes += all.size() * 8;
    stamp("sizes gathered");
    auto rows_of = [&](uint32_t src, uint32_t dst) { return all[(size_t)src * 2 * n + dst]; };
    auto keys_of = [&](uint32_t src, uint32_t dst) { return all[(size_t)src * 2 * n + n + dst]; };
    std::vector<uint64_t> s_bytes(n, 0), s_off(n, 0), r_bytes(n, 0), r_off(n, 0);
    uint64_t s_total = 0, r_total = 0;
    for (uint32_t p = 0; p < n; ++p) {
        s_bytes[p] = (p == rank || rows_of(rank, p) == 0) ? 0 : chunk_bytes_for(rows_of(rank, p), keys_of(rank, p));
        s_off[p] = s_total; s_total += s_bytes[p];
        r_bytes[p] = (p == rank || rows_of(p, rank) == 0) ? 0 : chunk_bytes_for(rows_of(p, rank), keys_of(p, rank));
        r_off[p] = r_total; r_total += r_bytes[p];
    }
    if ((rc = c->m_send.ensure(s_total ? s_total : 16))) return rc;
    if ((rc = c->m_recv.ensure(r_total ? r_total : 16))) return rc;
    const uint64_t before = g_launches;
    if (s_total && (rc = vfb_internal_partition_fill(c, n, rank, true, c->m_send.as<uint8_t>(), s_off.data()))) return rc;
    stamp("chunks filled");
    VFB_NCCL(a, a->GroupStart());
    for (uint32_t k = 1; k < n; ++k) {
        const uint32_t to = (rank + k) % n, from = (rank + n - k) % n;
        if (s_bytes[to]) VFB_NCCL(a, a->Send(c->m_send.as<uint8_t>() + s_off[to], (size_t)s_bytes[to], NCCL_UINT8, (int)to, (nccl_comm)comm, c->st_compute));
        if (r_bytes[from]) VFB_NCCL(a, a->Recv(c->m_recv.as<uint8_t>() + r_off[from], (size_t)r_bytes[from], NCCL_UINT8, (int)from, (nccl_comm)comm, c->st_compute));
    }
    VFB_NCCL(a, a->GroupEnd());
    bump_launches_for(c, before);
    stamp("chunks exchanged");
    for (uint32_t p = 0; p < n; ++p)
        if (r_bytes[p] && (rc = vfb_internal_absorb_known(c, c->m_recv.as<uint8_t>() + r_off[p], rows_of(p, rank), keys_of(p, rank)))) return rc;
    stamp("absorbed");
    if (tr) trace("merge_nccl rank %u: sent %.1f MB, received %.1f MB", rank, s_total / 1e6, r_total / 1e6);
    return VFB_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------ one process, n devices
struct vfb_multi {
    std::vector<vfb_ctx *> ctx;
    bool peers_enabled = false;
    PinBuf h_offsets, h_counts, h_data;     // the merged result columns
};

extern "C" {

int vfb_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int vfb_multi_create(const vfb_params *p, const int32_t *devices, uint32_t n_devices, vfb_multi **out)
{
    if (!p || !out) { set_error("null argument"); return VFB_ERR_ARG; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        set_error("no CUDA device available (this library has no CPU fallback)");
        return VFB_ERR_CUDA;
    }
    std::vector<int32_t> devs;
    if (!devices || n_devices == 0) for (int d = 0; d < ndev; ++d) devs.push_back(d);      // all visible devices
    else devs.assign(devices, devices + n_devices);
    for (size_t i = 0; i < devs.size(); ++i) {
        if (devs[i] < 0 || devs[i] >= ndev) { set_error("no such CUDA device: " + std::to_string(devs[i])); return VFB_ERR_ARG; }
        // (tests on a one-GPU box run two contexts on the same device: VFB_MULTI_ALLOW_DUP=1)
        for (size_t j = 0; j < i && !getenv("VFB_MULTI_ALLOW_DUP"); ++j)
            if (devs[j] == devs[i]) { set_error("a device is listed twice"); return VFB_ERR_ARG; }
    }
    vfb_multi *m = new vfb_multi;
    for (int32_t d : devs) {
        vfb_params q = *p;
        q.device = d;
        vfb_ctx *c = nullptr;
        const int rc = vfb_create(&q, &c);
        if (rc) {
            const std::string keep = vfb_last_error();
            vfb_multi_destroy(m);
            set_error(keep);
            return rc;
        }
        m->ctx.push_back(c);
    }
    *out = m;
    return VFB_OK;
}

int vfb_multi_destroy(vfb_multi *m)
{
    if (!m) return VFB_OK;
    for (vfb_ctx *c : m->ctx) vfb_destroy(c);
    m->h_offsets.release(); m->h_counts.release(); m->h_data.release();
    delete m;
    return VFB_OK;
}

uint32_t vfb_multi_devices(const vfb_multi *m) { return m ? (uint32_t)m->ctx.size() : 0; }

vfb_ctx *vfb_multi_ctx(vfb_multi *m, uint32_t i) { return (m && i < m->ctx.size()) ? m->ctx[i] : nullptr; }

int vfb_multi_run_file(vfb_multi *m, const char *path, uint32_t flags, uint64_t *n_reads)
{
    if (!m || !path || m->ctx.empty()) { set_error("null argument"); return VFB_ERR_ARG; }
    return vfb_internal_run_file(m->ctx.data(), (uint32_t)m->ctx.size(), path, flags, n_reads);
}

int vfb_multi_set_progress(vfb_multi *m, vfb_progress_fn fn, void *user)
{
    if (!m || m->ctx.empty()) { set_error("null argument"); return VFB_ERR_ARG; }
    return vfb_set_progress(m->ctx[0], fn, user);
}

int vfb_multi_sync(vfb_multi *m)
{
    if (!m) { set_error("null argument"); return VFB_ERR_ARG; }
    for (vfb_ctx *c : m->ctx) { const int rc = vfb_sync(c); if (rc) return rc; }
    return VFB_OK;
}

int vfb_multi_reset(vfb_multi *m)
{
    if (!m) { set_error("null argument"); return VFB_ERR_ARG; }
    for (vfb_ctx *c : m->ctx) { const int rc = vfb_reset(c); if (rc) return rc; }
    return VFB_OK;
}

// All-to-all over peer copies: afterwards context i holds exactly the keys it owns, with global counts.
int vfb_multi_merge(vfb_multi *m)
{
    if (!m) { set_error("null argument"); return VFB_ERR_ARG; }
    const uint32_t n = (uint32_t)m->ctx.size();
    if (n <= 1) return VFB_OK;
    int rc;
    if (!m->peers_enabled) {
        // direct NVLink paths where the topology has them (a copy between devices without peer access is staged
        // through the host by the driver: slower, still correct)
        for (uint32_t i = 0; i < n; ++i) {
            VFB_CUDA(cudaSetDevice(m->ctx[i]->device));
            for (uint32_t j = 0; j < n; ++j) {
                if (i == j) continue;
                int can = 0;
                if (cudaDeviceCanAccessPeer(&can, m->ctx[i]->device, m->ctx[j]->device) == cudaSuccess && can) {
                    const cudaError_t e = cudaDeviceEnablePeerAccess(m->ctx[j]->device, 0);
                    if (e != cudaSuccess) cudaGetLastError();      // already enabled is fine
                } else cudaGetLastError();
            }
        }
        m->peers_enabled = true;
    }
    // export on every device (kernels of different devices run side by side; the size fetch synchronises each)
    std::vector<std::vector<uint64_t>> bytes(n, std::vector<uint64_t>(n)), offs(n, std::vector<uint64_t>(n)),
        rows(n, std::vector<uint64_t>(n)), keys(n, std::vector<uint64_t>(n));
    for (uint32_t i = 0; i < n; ++i)
        if ((rc = vfb_internal_merge_export(m->ctx[i], n, i, true, bytes[i].data(), offs[i].data(), rows[i].data(), keys[i].data()))) return rc;
    // every destination pulls its chunks and absorbs them on its own compute stream
    for (uint32_t r = 0; r < n; ++r) {
        vfb_ctx *dst = m->ctx[r];
        uint64_t total = 0;
        std::vector<uint64_t> roff(n, 0);
        for (uint32_t i = 0; i < n; ++i) { roff[i] = total; total += bytes[i][r]; }
        VFB_CUDA(cudaSetDevice(dst->device));
        if ((rc = dst->m_recv.ensure(total ? total : 16))) return rc;
        for (uint32_t k = 1; k < n; ++k) {
            const uint32_t i = (r + k) % n;                 // staggered sources: no two destinations start on one source
            if (!bytes[i][r]) continue;
            vfb_ctx *src = m->ctx[i];
            VFB_CUDA(cudaStreamWaitEvent(dst->st_compute, src->m_filled, 0));
            VFB_CUDA(cudaMemcpyPeerAsync(dst->m_recv.as<uint8_t>() + roff[i], dst->device, src->m_send.as<uint8_t>() + offs[i][r],
                                         src->device, bytes[i][r], dst->st_compute));
            if ((rc = vfb_internal_absorb_known(dst, dst->m_recv.as<uint8_t>() + roff[i], rows[i][r], keys[i][r]))) return rc;
        }
    }
    // a send buffer may be refilled only after every peer has copied out of it
    return vfb_multi_sync(m);
}

int vfb_multi_get_stats(vfb_multi *m, vfb_stats *out)
{
    if (!m || !out) { set_error("null argument"); return VFB_ERR_ARG; }
    memset(out, 0, sizeof *out);
    for (size_t i = 0; i < m->ctx.size(); ++i) {
        vfb_stats s;
        const int rc = vfb_get_stats(m->ctx[i], &s);
        if (rc) return rc;
        out->reads += s.reads; out->dp_prefix += s.dp_prefix; out->dp_suffix += s.dp_suffix; out->dp_cells += s.dp_cells;
        out->counted += s.counted; out->unique += s.unique; out->text_bytes += s.text_bytes;
        out->kernel_launches += s.kernel_launches; out->h2d_bytes += s.h2d_bytes; out->d2h_bytes += s.d2h_bytes;
        out->ms_scan += s.ms_scan; out->ms_worklist += s.ms_worklist; out->ms_dp += s.ms_dp; out->ms_translate += s.ms_translate;
        out->ms_count += s.ms_count; out->ms_total += s.ms_total; out->dp_kernel_launches += s.dp_kernel_launches;
        out->dp_kernel_kind = s.dp_kernel_kind; out->dp_cells_computed += s.dp_cells_computed; out->dp_windows += s.dp_windows;
        out->ms_dp_filter += s.ms_dp_filter; out->ms_dp_window += s.ms_dp_window;
        out->reverse_reads += s.reverse_reads; out->reverse_counted += s.reverse_counted;
    }
    return VFB_OK;
}

// Merge, then every device writes its partition into its piece of one set of pinned host columns.
static int multi_export(vfb_multi *m, uint64_t *rows_out, uint64_t *bytes_out)
{
    int rc = vfb_multi_merge(m);
    if (rc) return rc;
    const size_t n = m->ctx.size();
    std::vector<uint64_t> rows(n), bytes(n);
    uint64_t tr = 0, tb = 0;
    for (size_t i = 0; i < n; ++i) {
        if ((rc = vfb_internal_export_sizes(m->ctx[i], &rows[i], &bytes[i]))) return rc;
        tr += rows[i]; tb += bytes[i];
    }
    if ((rc = m->h_offsets.ensure((tr + 1) * 8))) return rc;
    if ((rc = m->h_counts.ensure((tr ? tr : 1) * 8))) return rc;
    if ((rc = m->h_data.ensure(tb ? tb : 16))) return rc;
    uint64_t r0 = 0, b0 = 0;
    for (size_t i = 0; i < n; ++i) {
        if ((rc = vfb_internal_export_write(m->ctx[i], b0, (uint64_t *)m->h_offsets.p + r0, (uint64_t *)m->h_counts.p + r0,
                                            (uint8_t *)m->h_data.p + b0))) return rc;
        r0 += rows[i]; b0 += bytes[i];
    }
    if ((rc = vfb_multi_sync(m))) return rc;
    ((uint64_t *)m->h_offsets.p)[tr] = tb;
    *rows_out = tr; *bytes_out = tb;
    return VFB_OK;
}

int vfb_multi_finish(vfb_multi *m, vfb_table *out)
{
    if (!m || !out || m->ctx.empty()) { set_error("null argument"); return VFB_ERR_ARG; }
    memset(out, 0, sizeof *out);
    uint64_t rows = 0, bytes = 0;
    const int rc = multi_export(m, &rows, &bytes);
    if (rc) return rc;
    out->rows = rows; out->key_bytes = bytes;
    out->offsets = (uint64_t *)m->h_offsets.p;
    out->counts = (uint64_t *)m->h_counts.p;
    out->data = (uint8_t *)m->h_data.p;
    out->owner = m;
    return VFB_OK;
}

int vfb_multi_finish_arrow(vfb_multi *m, vfb_arrow_array *out_array, vfb_arrow_schema *out_schema)
{
    if (!m || !out_array || !out_schema || m->ctx.empty()) { set_error("null argument"); return VFB_ERR_ARG; }
    uint64_t rows = 0, bytes = 0;
    const int rc = multi_export(m, &rows, &bytes);
    if (rc) return rc;
    PinBuf o = m->h_offsets, d = m->h_data, n = m->h_counts;
    m->h_offsets = PinBuf(); m->h_data = PinBuf(); m->h_counts = PinBuf();
    return vfb_internal_arrow_wrap(o, d, n, rows, out_array, out_schema);
}

}  // extern "C"
