// C-ABI glue: error strings, device upload of the tables, the host-buffer entry
// point (pinned/pageable GAF bytes -> chunked H2D overlapped with the filter
// kernel -> counts, stats and hits back on the host) and the
// informative_aln.json writer (filter-alignments.py:174-175).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <thread>

#include "svjg_internal.h"

namespace svjg {

static thread_local std::string g_err;

int set_error(int code, const std::string &msg) {
    g_err = msg;
    return code;
}
int cuda_fail(int cuda_err, const char *what) {
    g_err = std::string("CUDA error: ") + cudaGetErrorString(cudaError_t(cuda_err)) + " in " + what;
    return SVJG_E_CUDA;
}

// ---------------------------------------------------------------------------
// workspace of svjg_filter_host
// ---------------------------------------------------------------------------
struct HostWs {
    static constexpr uint64_t CHUNK = 64ull << 20;
    uint8_t *d_buf[2] = {nullptr, nullptr};
    uint64_t buf_cap = 0;
    uint32_t *d_counts = nullptr;
    svjg_filter_stats *d_stats = nullptr;
    uint32_t *d_hit[3] = {nullptr, nullptr, nullptr};
    uint64_t hit_cap = 0;
    cudaStream_t s_copy = nullptr, s_comp = nullptr;
    cudaEvent_t copied[2] = {nullptr, nullptr}, freed[2] = {nullptr, nullptr};
    uint64_t *d_off64 = nullptr;              // absolute hit offsets (written by the kernels)
    // svjg_filter_json_host: the whole file resident, the text it renders, and the page-locked copy the caller reads
    uint8_t *d_all = nullptr;
    uint64_t all_cap = 0;
    char *h_json = nullptr;
    uint64_t json_cap = 0;
    uint64_t hits_per_gib = 0;                // what the last file needed: the first guess for the next one
    bool pending = false;                     // svjg_filter_json_begin done, svjg_filter_json_finish to come
    uint64_t pending_hits = 0;
    uint64_t range_base = 0;                  // file offset of the bytes in d_all (svjg_filter_json_begin_at)
    LineSrc src{};                            // where the renderer finds the lines: d_all, or several devices' after a gather
    // svjg_filter_json_write: two slices of the text on the device and two page-locked ones on the host
    uint8_t *d_slice[2] = {nullptr, nullptr};
    char *h_slice[2] = {nullptr, nullptr};
    uint64_t slice_cap = 0;
};

void free_host_ws(svjg_tables *t) {
    HostWs *w = t->ws;
    if (!w) return;
    for (int i = 0; i < 2; ++i) {
        if (w->d_buf[i]) cudaFree(w->d_buf[i]);
        if (w->copied[i]) cudaEventDestroy(w->copied[i]);
        if (w->freed[i]) cudaEventDestroy(w->freed[i]);
    }
    for (int i = 0; i < 3; ++i)
        if (w->d_hit[i]) cudaFree(w->d_hit[i]);
    if (w->d_counts) cudaFree(w->d_counts);
    if (w->d_stats) cudaFree(w->d_stats);
    if (w->d_off64) cudaFree(w->d_off64);
    if (w->d_all) cudaFree(w->d_all);
    if (w->h_json) cudaFreeHost(w->h_json);
    for (int i = 0; i < 2; ++i) {
        if (w->d_slice[i]) cudaFree(w->d_slice[i]);
        if (w->h_slice[i]) cudaFreeHost(w->h_slice[i]);
    }
    if (w->s_copy) cudaStreamDestroy(w->s_copy);
    if (w->s_comp) cudaStreamDestroy(w->s_comp);
    delete w;
    t->ws = nullptr;
}

}  // namespace svjg

using namespace svjg;

extern "C" const char *svjg_version(void) { return "svjg-b200 0.1.0 (sm_100a)"; }
extern "C" const char *svjg_last_error(void) { return g_err.c_str(); }

// page-locked host memory without a tensor library (file buffers of the command-line front-ends)
extern "C" int svjg_host_alloc(uint64_t bytes, void **out) {
    if (!out) return set_error(SVJG_E_ARG, "svjg_host_alloc: NULL argument");
    SVJG_CUDA(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
    return SVJG_OK;
}
extern "C" int svjg_host_free(void *p) {
    if (p) SVJG_CUDA(cudaFreeHost(p));
    return SVJG_OK;
}
// page-lock / release memory the caller already owns (e.g. a file read while the context was created)
extern "C" int svjg_host_register(void *p, uint64_t bytes) {
    if (!p || !bytes) return SVJG_OK;
    SVJG_CUDA(cudaHostRegister(p, bytes, cudaHostRegisterDefault));
    return SVJG_OK;
}
extern "C" int svjg_host_unregister(void *p) {
    if (p) SVJG_CUDA(cudaHostUnregister(p));
    return SVJG_OK;
}
// creates the CUDA context of `device` (about a second): call it from a thread while the host reads files
extern "C" int svjg_device_init(int device) {
    SVJG_CUDA(cudaSetDevice(device));
    SVJG_CUDA(cudaFree(nullptr));
    return SVJG_OK;
}

// Text-mode line ends (filter-alignments.py:123 reads the GAF in text mode): "\r\n" and a lone "\r" become "\n".
// In place, one pass; returns the new length.
extern "C" uint64_t svjg_translate_newlines(uint8_t *p, uint64_t n) {
    if (!p) return 0;
    uint8_t *cr = static_cast<uint8_t *>(memchr(p, '\r', n));
    if (!cr) return n;
    uint64_t r = uint64_t(cr - p), w = r;
    while (r < n) {
        if (p[r] == '\r') {
            p[w++] = '\n';
            r += (r + 1 < n && p[r + 1] == '\n') ? 2 : 1;
            continue;
        }
        // copy the run up to the next carriage return in one go
        const uint8_t *nx = static_cast<const uint8_t *>(memchr(p + r, '\r', n - r));
        const uint64_t run = nx ? uint64_t(nx - (p + r)) : n - r;
        if (w != r) memmove(p + w, p + r, run);
        w += run;
        r += run;
    }
    return w;
}

extern "C" int svjg_tables_to_device(svjg_tables *t, int device) {
    if (!t) return set_error(SVJG_E_ARG, "svjg_tables_to_device: NULL tables");
    if (t->device == device) return SVJG_OK;
    if (t->device >= 0) return set_error(SVJG_E_ARG, "tables already live on another device");
    SVJG_CUDA(cudaSetDevice(device));
    auto up = [&](void **dst, const void *src, size_t bytes) -> cudaError_t {
        cudaError_t e = cudaMalloc(dst, bytes ? bytes : 16);
        if (e != cudaSuccess) return e;
        return bytes ? cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice) : cudaSuccess;
    };
    SVJG_CUDA(up(&t->d_links, t->links.data(), t->links.size() * sizeof(LinkSlot)));
    SVJG_CUDA(up(&t->d_nodes, t->nodes.data(), t->nodes.size() * sizeof(NodeSlot)));
    SVJG_CUDA(up(&t->d_blob, t->blob.data(), t->blob.size()));
    SVJG_CUDA(up(&t->d_entries, t->entries.data(), t->entries.size() * sizeof(uint32_t)));
    SVJG_CUDA(up(&t->d_pnodes, t->pnodes.data(), t->pnodes.size() * sizeof(PNodeSlot)));
    t->dev.pnodes = static_cast<const PNodeSlot *>(t->d_pnodes);
    t->dev.pnode_mask = uint32_t(t->pnodes.size() - 1);
    t->dev.links = static_cast<const LinkSlot *>(t->d_links);
    t->dev.nodes = static_cast<const NodeSlot *>(t->d_nodes);
    t->dev.blob = static_cast<const uint8_t *>(t->d_blob);
    t->dev.entries = static_cast<const uint32_t *>(t->d_entries);
    t->dev.link_mask = uint32_t(t->links.size() - 1);
    t->dev.node_mask = uint32_t(t->nodes.size() - 1);
    t->dev.num_sv = uint32_t(t->sv_ids.size());
    t->device = device;
    return SVJG_OK;
}

extern "C" void svjg_tables_free(svjg_tables *t) {
    if (!t) return;
    if (t->device >= 0) {
        cudaSetDevice(t->device);
        free_host_ws(t);
        free_json_keys(t);
        cudaFree(t->d_links);
        cudaFree(t->d_nodes);
        cudaFree(t->d_blob);
        cudaFree(t->d_entries);
        cudaFree(t->d_pnodes);
    }
    delete t;
}

// ---------------------------------------------------------------------------
// host-buffer filter
// ---------------------------------------------------------------------------
static int ensure_ws(svjg_tables *t, uint32_t num_sv) {
    if (t->ws) return SVJG_OK;
    t->ws = new HostWs();
    HostWs *w = t->ws;
    SVJG_CUDA(cudaStreamCreateWithFlags(&w->s_copy, cudaStreamNonBlocking));
    SVJG_CUDA(cudaStreamCreateWithFlags(&w->s_comp, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
        SVJG_CUDA(cudaEventCreateWithFlags(&w->copied[i], cudaEventDisableTiming));
        SVJG_CUDA(cudaEventCreateWithFlags(&w->freed[i], cudaEventDisableTiming));
    }
    SVJG_CUDA(cudaMalloc(&w->d_counts, std::max<size_t>(16, size_t(num_sv) * 8)));
    SVJG_CUDA(cudaMalloc(&w->d_stats, sizeof(svjg_filter_stats)));
    return SVJG_OK;
}

static int ensure_hit_arrays(HostWs *w, uint64_t hit_cap) {
    if (w->hit_cap >= hit_cap) return SVJG_OK;
    for (int i = 0; i < 3; ++i) {
        if (w->d_hit[i]) SVJG_CUDA(cudaFree(w->d_hit[i]));
        w->d_hit[i] = nullptr;
    }
    if (w->d_off64) SVJG_CUDA(cudaFree(w->d_off64));
    w->d_off64 = nullptr;
    w->hit_cap = 0;
    for (int i = 0; i < 3; ++i) SVJG_CUDA(cudaMalloc(&w->d_hit[i], hit_cap * 4));
    SVJG_CUDA(cudaMalloc(&w->d_off64, hit_cap * 8));
    w->hit_cap = hit_cap;
    return SVJG_OK;
}

// Host bytes through the filter chain into d_counts and w->d_stats (neither is reset here), on w->s_comp: chunks cut
// at line ends, each copied on w->s_copy into one of two device buffers while the kernels work on the other.
// Returns once every chunk is enqueued.
static int filter_chunks(svjg_tables *t, const uint8_t *gaf, uint64_t n_bytes, int64_t d_over, uint32_t *d_counts,
                         uint32_t *k_sv2, uint64_t *k_off, uint32_t *k_len, uint64_t hit_cap) {
    HostWs *w = t->ws;
    // chunk plan: cut at line ends, each chunk < 4 GiB
    std::vector<uint64_t> cut{0};
    while (cut.back() < n_bytes) {
        uint64_t b = cut.back(), e = std::min(n_bytes, b + HostWs::CHUNK);
        if (e < n_bytes) {
            const void *nl = memrchr(gaf + b, '\n', size_t(e - b));
            if (nl) {
                e = uint64_t(static_cast<const uint8_t *>(nl) - gaf) + 1;
            } else {
                const void *fw = memchr(gaf + e, '\n', size_t(n_bytes - e));
                e = fw ? uint64_t(static_cast<const uint8_t *>(fw) - gaf) + 1 : n_bytes;
            }
        }
        if (e - b >= 0xFFFF0000ull) return set_error(SVJG_E_ARG, "a single GAF line exceeds 4 GiB");
        cut.push_back(e);
    }
    const size_t n_chunks = cut.size() - 1;
    uint64_t max_chunk = 0;
    for (size_t k = 0; k < n_chunks; ++k) max_chunk = std::max(max_chunk, cut[k + 1] - cut[k]);

    if (w->buf_cap < max_chunk) {
        for (int i = 0; i < 2; ++i) {
            if (w->d_buf[i]) SVJG_CUDA(cudaFree(w->d_buf[i]));
            w->d_buf[i] = nullptr;
        }
        w->buf_cap = 0;
        uint64_t cap = (max_chunk + 255) & ~255ull;
        for (int i = 0; i < (n_chunks > 1 ? 2 : 1); ++i) SVJG_CUDA(cudaMalloc(&w->d_buf[i], cap));
        w->buf_cap = cap;
    } else if (n_chunks > 1 && !w->d_buf[1]) {
        SVJG_CUDA(cudaMalloc(&w->d_buf[1], w->buf_cap));
    }
    for (size_t k = 0; k < n_chunks; ++k) {
        int b = int(k & 1);
        uint64_t len = cut[k + 1] - cut[k];
        if (k >= 2) SVJG_CUDA(cudaStreamWaitEvent(w->s_copy, w->freed[b], 0));
        SVJG_CUDA(cudaMemcpyAsync(w->d_buf[b], gaf + cut[k], len, cudaMemcpyHostToDevice, w->s_copy));
        SVJG_CUDA(cudaEventRecord(w->copied[b], w->s_copy));
        SVJG_CUDA(cudaStreamWaitEvent(w->s_comp, w->copied[b], 0));
        int rc = filter_device_abs(t, w->d_buf[b], len, cut[k], d_over, d_counts, k_sv2, nullptr, k_off, k_len, hit_cap,
                                   w->d_stats, w->s_comp);
        if (rc) {
            // copies out of the caller's buffer and kernels may still be in flight: not behind the caller's back
            cudaStreamSynchronize(w->s_copy);
            cudaStreamSynchronize(w->s_comp);
            return rc;
        }
        SVJG_CUDA(cudaEventRecord(w->freed[b], w->s_comp));
    }
    return SVJG_OK;
}

// the stats of a finished filter call: SVJG_E_INPUT where the reference would raise
static int input_status(svjg_filter_stats *stats, uint64_t n_bytes) {
    if (n_bytes == 0) memset(stats, 0, sizeof *stats), stats->err_offset = ~0ull;
    if (stats->status) {
        char msg[160];
        snprintf(msg, sizeof msg, "GAF line at byte %llu: the reference raises here (reason %llu)",
                 (unsigned long long)stats->err_offset, (unsigned long long)stats->status);
        return set_error(SVJG_E_INPUT, msg);
    }
    return SVJG_OK;
}

extern "C" int svjg_filter_host(svjg_tables *t, const uint8_t *gaf, uint64_t n_bytes, int64_t d_over, uint32_t *counts,
                                uint32_t *hit_sv2, uint64_t *hit_off, uint32_t *hit_len, uint64_t hit_cap,
                                svjg_filter_stats *stats) {
    if (!t || t->device < 0) return set_error(SVJG_E_ARG, "svjg_filter_host: tables are not on a device");
    if (!counts || !stats || (n_bytes && !gaf)) return set_error(SVJG_E_ARG, "svjg_filter_host: NULL argument");
    if (hit_cap && (!hit_sv2 || !hit_off || !hit_len)) return set_error(SVJG_E_ARG, "svjg_filter_host: NULL hit buffer");
    SVJG_CUDA(cudaSetDevice(t->device));
    const uint32_t num_sv = uint32_t(t->sv_ids.size());

    int rc = ensure_ws(t, num_sv);
    if (rc) return rc;
    HostWs *w = t->ws;
    rc = ensure_hit_arrays(w, hit_cap);
    if (rc) return rc;
    // Result arrays in page-locked host memory are written by the kernels themselves (the device can
    // address them): the hits cross PCIe while later chunks are still coming in, and no copy is left
    // for the end.  Pageable arrays get the hits by a copy from device buffers.
    auto device_view = [](void *p) -> void * {
        cudaPointerAttributes at;
        if (!p || cudaPointerGetAttributes(&at, p) != cudaSuccess) {
            cudaGetLastError();
            return nullptr;
        }
        return at.type == cudaMemoryTypeHost ? at.devicePointer : nullptr;
    };
    uint32_t *k_sv2 = w->d_hit[0], *k_len = w->d_hit[2];
    uint64_t *k_off = w->d_off64;
    bool direct = false;
    // Up to 64 MB of hit tuples; beyond that the copy engines take them at the end.  (Measured: 0.5 GB
    // of tuples per GPU written by the kernels is fine on one GPU -- 5 ms, hidden behind the upload --
    // but took 1.3 s when eight GPUs of a node did it at once.)
    if (hit_cap && hit_cap * 16 <= (64ull << 20)) {
        void *v0 = device_view(hit_sv2), *v1 = device_view(hit_off), *v2 = device_view(hit_len);
        if (v0 && v1 && v2) {
            k_sv2 = static_cast<uint32_t *>(v0);
            k_off = static_cast<uint64_t *>(v1);
            k_len = static_cast<uint32_t *>(v2);
            direct = true;
        }
    }

    rc = svjg_filter_reset(w->d_counts, num_sv, w->d_stats, w->s_comp);
    if (rc) return rc;
    rc = filter_chunks(t, gaf, n_bytes, d_over, w->d_counts, k_sv2, k_off, k_len, hit_cap);
    if (rc) return rc;
    SVJG_CUDA(cudaMemcpyAsync(stats, w->d_stats, sizeof(svjg_filter_stats), cudaMemcpyDeviceToHost, w->s_comp));
    SVJG_CUDA(cudaMemcpyAsync(counts, w->d_counts, size_t(num_sv) * 8, cudaMemcpyDeviceToHost, w->s_comp));
    SVJG_CUDA(cudaStreamSynchronize(w->s_comp));
    rc = input_status(stats, n_bytes);
    if (rc) return rc;
    if (hit_cap == 0) return SVJG_OK;
    if (stats->n_hits > hit_cap) return set_error(SVJG_E_HITS_OVERFLOW, "hit buffers too small");
    const uint64_t nh = stats->n_hits;
    if (nh && !direct) {
        // pageable result arrays: staged by the driver
        SVJG_CUDA(cudaMemcpyAsync(hit_sv2, w->d_hit[0], nh * 4, cudaMemcpyDeviceToHost, w->s_comp));
        SVJG_CUDA(cudaMemcpyAsync(hit_off, w->d_off64, nh * 8, cudaMemcpyDeviceToHost, w->s_comp));
        SVJG_CUDA(cudaMemcpyAsync(hit_len, w->d_hit[2], nh * 4, cudaMemcpyDeviceToHost, w->s_comp));
        SVJG_CUDA(cudaStreamSynchronize(w->s_comp));
    }
    return SVJG_OK;
}

// ---------------------------------------------------------------------------
// cohort counters: one slice per sample, filled by the same chunk loop
// ---------------------------------------------------------------------------
extern "C" int svjg_cohort_create(svjg_tables *t, uint32_t n_samples, svjg_cohort **out) {
    if (!t || t->device < 0) return set_error(SVJG_E_ARG, "svjg_cohort_create: tables are not on a device");
    if (!out || n_samples == 0) return set_error(SVJG_E_ARG, "svjg_cohort_create: bad argument");
    SVJG_CUDA(cudaSetDevice(t->device));
    svjg_cohort *c = new svjg_cohort();
    c->t = t;
    c->n_samples = n_samples;
    c->num_sv = uint32_t(t->sv_ids.size());
    const size_t bytes = std::max<size_t>(16, size_t(n_samples) * c->num_sv * 8);
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMalloc(&c->d_counts, bytes);
    if (e == cudaSuccess) e = cudaMemset(c->d_counts, 0, bytes);
    if (e != cudaSuccess) {
        svjg_cohort_free(c);
        return cuda_fail(int(e), "svjg_cohort_create");
    }
    *out = c;
    return SVJG_OK;
}

extern "C" void svjg_cohort_free(svjg_cohort *c) {
    if (!c) return;
    cudaSetDevice(c->t->device);
    if (c->d_counts) cudaFree(c->d_counts);
    if (c->d_lut) cudaFree(c->d_lut);
    if (c->d_blk) cudaFree(c->d_blk);
    if (c->d_site) cudaFree(c->d_site);
    if (c->d_ploidy) cudaFree(c->d_ploidy);
    if (c->d_plw) cudaFree(c->d_plw);
    if (c->d_post) cudaFree(c->d_post);
    if (c->d_qc) cudaFree(c->d_qc);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

extern "C" int svjg_cohort_filter(svjg_cohort *c, uint32_t sample, const uint8_t *gaf, uint64_t n_bytes, int64_t d_over,
                                  svjg_filter_stats *stats) {
    if (!c || !stats || (n_bytes && !gaf)) return set_error(SVJG_E_ARG, "svjg_cohort_filter: NULL argument");
    if (sample >= c->n_samples) return set_error(SVJG_E_ARG, "svjg_cohort_filter: sample out of range");
    svjg_tables *t = c->t;
    SVJG_CUDA(cudaSetDevice(t->device));
    int rc = ensure_ws(t, c->num_sv);
    if (rc) return rc;
    HostWs *w = t->ws;
    uint32_t *d_counts = c->d_counts + size_t(sample) * c->num_sv * 2;
    rc = svjg_filter_reset(d_counts, 0, w->d_stats, w->s_comp);          // the stats only: the counters accumulate
    if (rc) return rc;
    rc = filter_chunks(t, gaf, n_bytes, d_over, d_counts, nullptr, nullptr, nullptr, 0);
    if (rc) return rc;
    SVJG_CUDA(cudaMemcpyAsync(stats, w->d_stats, sizeof(svjg_filter_stats), cudaMemcpyDeviceToHost, w->s_comp));
    SVJG_CUDA(cudaStreamSynchronize(w->s_comp));
    return input_status(stats, n_bytes);
}

extern "C" int svjg_cohort_read_counts(svjg_cohort *c, uint32_t sample, uint32_t *counts) {
    if (!c || (!counts && c->num_sv)) return set_error(SVJG_E_ARG, "svjg_cohort_read_counts: NULL argument");
    if (sample >= c->n_samples) return set_error(SVJG_E_ARG, "svjg_cohort_read_counts: sample out of range");
    SVJG_CUDA(cudaSetDevice(c->t->device));
    SVJG_CUDA(cudaMemcpyAsync(counts, c->d_counts + size_t(sample) * c->num_sv * 2, size_t(c->num_sv) * 8,
                              cudaMemcpyDeviceToHost, c->stream));
    SVJG_CUDA(cudaStreamSynchronize(c->stream));
    return SVJG_OK;
}

extern "C" int svjg_cohort_load_counts(svjg_cohort *c, uint32_t sample, const uint32_t *counts) {
    if (!c || (!counts && c->num_sv)) return set_error(SVJG_E_ARG, "svjg_cohort_load_counts: NULL argument");
    if (sample >= c->n_samples) return set_error(SVJG_E_ARG, "svjg_cohort_load_counts: sample out of range");
    SVJG_CUDA(cudaSetDevice(c->t->device));
    SVJG_CUDA(cudaMemcpyAsync(c->d_counts + size_t(sample) * c->num_sv * 2, counts, size_t(c->num_sv) * 8,
                              cudaMemcpyHostToDevice, c->stream));
    SVJG_CUDA(cudaStreamSynchronize(c->stream));
    return SVJG_OK;
}

// ---------------------------------------------------------------------------
// host-buffer filter with the informative_aln.json text rendered on the device
// ---------------------------------------------------------------------------
extern "C" int svjg_filter_json_begin(svjg_tables *t, const uint8_t *gaf, uint64_t n_bytes, int64_t d_over, uint32_t *counts,
                                      svjg_filter_stats *stats) {
    return svjg_filter_json_begin_at(t, gaf, n_bytes, 0, d_over, counts, stats);
}

extern "C" int svjg_filter_json_begin_at(svjg_tables *t, const uint8_t *gaf, uint64_t n_bytes, uint64_t base, int64_t d_over,
                                         uint32_t *counts, svjg_filter_stats *stats) {
    if (!t || t->device < 0) return set_error(SVJG_E_ARG, "svjg_filter_json_host: tables are not on a device");
    if (!counts || !stats || (n_bytes && !gaf)) return set_error(SVJG_E_ARG, "svjg_filter_json_host: NULL argument");
    SVJG_CUDA(cudaSetDevice(t->device));
    const uint32_t num_sv = uint32_t(t->sv_ids.size());
    if (int rc = ensure_ws(t, num_sv)) return rc;
    HostWs *w = t->ws;
    // the file stays on the device until its text is rendered: one buffer, filled chunk by chunk (cut at line
    // ends) while the chunks already there are filtered
    if (w->all_cap < n_bytes + 64) {
        if (w->d_all) SVJG_CUDA(cudaFree(w->d_all));
        w->d_all = nullptr;
        w->all_cap = 0;
        const uint64_t cap = ((n_bytes + 64) + (1ull << 20)) & ~((1ull << 20) - 1);
        // a file that does not fit beside its hits and its text: decline, svjg_filter_host streams it in chunks
        size_t mem_free = 0, mem_total = 0;
        SVJG_CUDA(cudaMemGetInfo(&mem_free, &mem_total));
        if (cap + cap / 2 > mem_free)
            return set_error(SVJG_E_UNSUPPORTED, "the file does not fit the device with its text: svjg_filter_host takes it in chunks");
        SVJG_CUDA(cudaMalloc(&w->d_all, cap));
        w->all_cap = cap;
    }
    std::vector<uint64_t> cut{0};
    while (cut.back() < n_bytes) {
        uint64_t b = cut.back(), e = std::min(n_bytes, b + HostWs::CHUNK);
        if (e < n_bytes) {
            const void *nl = memrchr(gaf + b, '\n', size_t(e - b));
            if (nl) {
                e = uint64_t(static_cast<const uint8_t *>(nl) - gaf) + 1;
            } else {
                const void *fw = memchr(gaf + e, '\n', size_t(n_bytes - e));
                e = fw ? uint64_t(static_cast<const uint8_t *>(fw) - gaf) + 1 : n_bytes;
            }
        }
        if (e - b >= 0xFFFF0000ull) return set_error(SVJG_E_ARG, "a single GAF line exceeds 4 GiB");
        cut.push_back(e);
    }
    const size_t n_chunks = cut.size() - 1;
    uint64_t guess = w->hits_per_gib ? (w->hits_per_gib * ((n_bytes >> 30) + 1) * 5) / 4 : n_bytes / 96;
    if (int rc = ensure_hit_arrays(w, std::max<uint64_t>(guess, 1u << 16))) return rc;

    cudaEvent_t up_done = w->copied[0];
    for (int attempt = 0;; ++attempt) {
        int rc = svjg_filter_reset(w->d_counts, num_sv, w->d_stats, w->s_comp);
        if (rc) return rc;
        for (size_t k = 0; k < n_chunks; ++k) {
            const uint64_t len = cut[k + 1] - cut[k];
            if (attempt == 0) {
                SVJG_CUDA(cudaMemcpyAsync(w->d_all + cut[k], gaf + cut[k], len, cudaMemcpyHostToDevice, w->s_copy));
                SVJG_CUDA(cudaEventRecord(up_done, w->s_copy));
                SVJG_CUDA(cudaStreamWaitEvent(w->s_comp, up_done, 0));
            }
            rc = filter_device_abs(t, w->d_all + cut[k], len, base + cut[k], d_over, w->d_counts, w->d_hit[0], nullptr, w->d_off64,
                                   w->d_hit[2], w->hit_cap, w->d_stats, w->s_comp, true);
            if (rc) {
                cudaStreamSynchronize(w->s_copy);
                cudaStreamSynchronize(w->s_comp);
                return rc;
            }
        }
        SVJG_CUDA(cudaMemcpyAsync(stats, w->d_stats, sizeof(svjg_filter_stats), cudaMemcpyDeviceToHost, w->s_comp));
        SVJG_CUDA(cudaStreamSynchronize(w->s_comp));
        if (n_bytes == 0) memset(stats, 0, sizeof *stats), stats->err_offset = ~0ull;
        if (stats->status) {
            char msg[160];
            snprintf(msg, sizeof msg, "GAF line at byte %llu: the reference raises here (reason %llu)",
                     (unsigned long long)stats->err_offset, (unsigned long long)stats->status);
            return set_error(SVJG_E_INPUT, msg);
        }
        if (stats->n_hits <= w->hit_cap) break;
        // more hits than there was room for: the file is resident, only the kernels run again
        if (attempt) return set_error(SVJG_E_HITS_OVERFLOW, "hit buffers too small");
        if (int rc2 = ensure_hit_arrays(w, stats->n_hits + 1024)) return rc2;
    }
    w->hits_per_gib = stats->n_hits / ((n_bytes >> 30) + 1);
    SVJG_CUDA(cudaMemcpyAsync(counts, w->d_counts, size_t(num_sv) * 8, cudaMemcpyDeviceToHost, w->s_comp));
    SVJG_CUDA(cudaStreamSynchronize(w->s_comp));
    w->pending_hits = stats->n_hits;
    w->pending = true;
    w->range_base = base;
    w->src = LineSrc{};
    w->src.n = 1;
    w->src.base[0] = w->d_all;
    w->src.start[0] = base;
    return SVJG_OK;
}

// Ranges of one file filtered on several devices (svjg_filter_json_begin_at, range k on ts[k], in file order): the hit
// tuples of devices 1.. are copied to device 0 (peer copies), the summed counters uploaded there, and the renderer of
// ts[0] (svjg_filter_json_finish / _write) reads every line where it lies -- its own memory or a peer's over NVLink.
extern "C" int svjg_filter_json_gather(svjg_tables **ts, int n, const uint32_t *counts_sum) {
    if (!ts || n < 1 || n > MAX_RANGES || !counts_sum) return set_error(SVJG_E_ARG, "svjg_filter_json_gather: bad argument");
    for (int d = 0; d < n; ++d)
        if (!ts[d] || !ts[d]->ws || !ts[d]->ws->pending || ts[d]->device < 0)
            return set_error(SVJG_E_ARG, "svjg_filter_json_gather: a device without svjg_filter_json_begin_at before it");
    HostWs *w0 = ts[0]->ws;
    const int dev0 = ts[0]->device;
    SVJG_CUDA(cudaSetDevice(dev0));
    uint64_t total = 0;
    for (int d = 0; d < n; ++d) {
        if (d && ts[d]->ws->range_base < ts[d - 1]->ws->range_base)
            return set_error(SVJG_E_ARG, "svjg_filter_json_gather: ranges out of file order");
        total += ts[d]->ws->pending_hits;
        if (d == 0 || ts[d]->device == dev0) continue;
        int can = 0;
        SVJG_CUDA(cudaDeviceCanAccessPeer(&can, dev0, ts[d]->device));
        if (!can) return set_error(SVJG_E_UNSUPPORTED, "no peer access between the devices: the host emitter writes the text");
        cudaError_t e = cudaDeviceEnablePeerAccess(ts[d]->device, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
        else if (e != cudaSuccess) return cuda_fail(int(e), "cudaDeviceEnablePeerAccess");
    }
    const uint64_t n0 = w0->pending_hits;
    if (w0->hit_cap < total) {
        // larger arrays that keep device 0's own tuples (sv2, offsets, lengths; d_hit[1] is not used on this route)
        uint32_t *sv2 = nullptr, *len = nullptr;
        uint64_t *off = nullptr;
        const uint64_t cap = total + 1024;
        cudaError_t me = cudaMalloc(&sv2, cap * 4);
        if (me == cudaSuccess) me = cudaMalloc(&len, cap * 4);
        if (me == cudaSuccess) me = cudaMalloc(&off, cap * 8);
        if (me != cudaSuccess) {
            cudaFree(sv2), cudaFree(len), cudaFree(off);        // cudaFree(NULL) is a no-op
            return cuda_fail(int(me), "svjg_filter_json_gather: hit arrays");
        }
        SVJG_CUDA(cudaMemcpyAsync(sv2, w0->d_hit[0], n0 * 4, cudaMemcpyDeviceToDevice, w0->s_comp));
        SVJG_CUDA(cudaMemcpyAsync(len, w0->d_hit[2], n0 * 4, cudaMemcpyDeviceToDevice, w0->s_comp));
        SVJG_CUDA(cudaMemcpyAsync(off, w0->d_off64, n0 * 8, cudaMemcpyDeviceToDevice, w0->s_comp));
        SVJG_CUDA(cudaStreamSynchronize(w0->s_comp));
        SVJG_CUDA(cudaFree(w0->d_hit[0]));
        SVJG_CUDA(cudaFree(w0->d_hit[2]));
        SVJG_CUDA(cudaFree(w0->d_off64));
        if (w0->d_hit[1]) SVJG_CUDA(cudaFree(w0->d_hit[1]));
        w0->d_hit[1] = nullptr;
        SVJG_CUDA(cudaMalloc(&w0->d_hit[1], cap * 4));
        w0->d_hit[0] = sv2, w0->d_hit[2] = len, w0->d_off64 = off;
        w0->hit_cap = cap;
    }
    LineSrc src{};
    src.n = uint32_t(n);
    uint64_t at = 0;
    for (int d = 0; d < n; ++d) {
        HostWs *w = ts[d]->ws;
        src.base[d] = w->d_all;
        src.start[d] = w->range_base;
        const uint64_t nh = w->pending_hits;
        if (d && nh) {
            SVJG_CUDA(cudaMemcpyPeerAsync(w0->d_hit[0] + at, dev0, w->d_hit[0], ts[d]->device, nh * 4, w0->s_comp));
            SVJG_CUDA(cudaMemcpyPeerAsync(w0->d_hit[2] + at, dev0, w->d_hit[2], ts[d]->device, nh * 4, w0->s_comp));
            SVJG_CUDA(cudaMemcpyPeerAsync(w0->d_off64 + at, dev0, w->d_off64, ts[d]->device, nh * 8, w0->s_comp));
        }
        at += nh;
        if (d) w->pending = false;
    }
    SVJG_CUDA(cudaMemcpyAsync(w0->d_counts, counts_sum, ts[0]->sv_ids.size() * 8, cudaMemcpyHostToDevice, w0->s_comp));
    SVJG_CUDA(cudaStreamSynchronize(w0->s_comp));
    w0->pending_hits = total;
    w0->src = src;
    return SVJG_OK;
}

extern "C" int svjg_filter_json_finish(svjg_tables *t, const char **json, uint64_t *json_len) {
    if (!t || !t->ws || !t->ws->pending) return set_error(SVJG_E_ARG, "svjg_filter_json_finish: no svjg_filter_json_begin before it");
    if (!json || !json_len) return set_error(SVJG_E_ARG, "svjg_filter_json_finish: NULL argument");
    SVJG_CUDA(cudaSetDevice(t->device));
    HostWs *w = t->ws;
    w->pending = false;
    uint8_t *d_text = nullptr;
    uint64_t len = 0;
    int rc = json_render_device(t, w->src, w->d_hit[0], w->d_off64, w->d_hit[2], w->pending_hits, w->d_counts, &d_text, &len, w->s_comp);
    if (rc) {
        cudaStreamSynchronize(w->s_comp);
        return rc;
    }
    if (w->json_cap < len) {
        if (w->h_json) cudaFreeHost(w->h_json);
        w->h_json = nullptr;
        w->json_cap = 0;
        const uint64_t cap = (len + len / 8 + (1ull << 20)) & ~((1ull << 20) - 1);
        cudaError_t e = cudaHostAlloc(reinterpret_cast<void **>(&w->h_json), cap, cudaHostAllocDefault);
        if (e != cudaSuccess) {
            cudaFreeAsync(d_text, w->s_comp);
            cudaStreamSynchronize(w->s_comp);
            return cuda_fail(int(e), "page-locked buffer for the JSON text");
        }
        w->json_cap = cap;
    }
    SVJG_CUDA(cudaMemcpyAsync(w->h_json, d_text, len, cudaMemcpyDeviceToHost, w->s_comp));
    SVJG_CUDA(cudaFreeAsync(d_text, w->s_comp));
    SVJG_CUDA(cudaStreamSynchronize(w->s_comp));
    *json = w->h_json;
    *json_len = len;
    return SVJG_OK;
}

// The second half for a text that goes to a file: rendered key range by key range into one of two device slices,
// copied to one of two page-locked slices and written from there by a thread of its own, so the slice behind it is
// rendered and copied meanwhile.  Neither side ever holds the whole text (it is 10 x the GAF where records sit
// in many lists); nothing is written where the renderer declines.
extern "C" int svjg_filter_json_write(svjg_tables *t, const char *path, uint64_t slice_bytes, uint64_t *json_len) {
    if (!t || !t->ws || !t->ws->pending) return set_error(SVJG_E_ARG, "svjg_filter_json_write: no svjg_filter_json_begin before it");
    if (!path) return set_error(SVJG_E_ARG, "svjg_filter_json_write: NULL path");
    SVJG_CUDA(cudaSetDevice(t->device));
    HostWs *w = t->ws;
    w->pending = false;
    if (!slice_bytes) slice_bytes = 64ull << 20;
    JsonPlan *plan = nullptr;
    if (int rc = json_plan(t, w->src, w->d_hit[0], w->d_off64, w->d_hit[2], w->pending_hits, w->d_counts, &plan, w->s_comp)) {
        cudaStreamSynchronize(w->s_comp);
        return rc;
    }
    const uint32_t num_sv = json_plan_keys(plan);
    std::vector<uint64_t> pos(size_t(num_sv) + 1), first_hit(size_t(num_sv) + 1);
    int rc = json_plan_key_positions(plan, pos.data(), first_hit.data(), w->s_comp);
    struct Slice {
        uint32_t lo, hi;
        uint64_t len;
    };
    std::vector<Slice> slices;
    uint64_t max_len = 2;
    if (!rc) {
        // whole keys per slice, as many as fit slice_bytes (a key with more text than that is a slice of its own);
        // the slice with the last key carries the two closing bytes
        uint32_t lo = 0;
        do {
            uint32_t hi = uint32_t(std::upper_bound(pos.begin() + lo, pos.end(), pos[lo] + slice_bytes) - pos.begin()) - 1;
            if (hi <= lo) hi = lo + 1;
            if (hi > num_sv) hi = num_sv;
            slices.push_back({lo, hi, pos[hi] - pos[lo] + (hi == num_sv ? 2u : 0u)});
            max_len = std::max(max_len, slices.back().len);
            lo = hi;
        } while (lo < num_sv);
        if (w->slice_cap < max_len) {
            for (int i = 0; i < 2 && !rc; ++i) {
                if (w->d_slice[i]) cudaFree(w->d_slice[i]);
                if (w->h_slice[i]) cudaFreeHost(w->h_slice[i]);
                w->d_slice[i] = nullptr, w->h_slice[i] = nullptr;
            }
            w->slice_cap = 0;
            for (int i = 0; i < 2 && !rc; ++i) {
                cudaError_t e = cudaMalloc(&w->d_slice[i], max_len);
                if (e == cudaSuccess) e = cudaHostAlloc(reinterpret_cast<void **>(&w->h_slice[i]), max_len, cudaHostAllocDefault);
                if (e != cudaSuccess) rc = cuda_fail(int(e), "svjg_filter_json_write: slice buffers");
            }
            if (!rc) w->slice_cap = max_len;
        }
    }
    FILE *f = rc ? nullptr : fopen(path, "wb");
    if (!rc && !f) rc = set_error(SVJG_E_IO, std::string("cannot write ") + path);
    if (rc) {
        json_plan_free(plan, w->s_comp);
        cudaStreamSynchronize(w->s_comp);
        return rc;
    }
    cudaEvent_t rendered[2], copied[2];
    for (int i = 0; i < 2; ++i) {
        cudaEventCreateWithFlags(&rendered[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&copied[i], cudaEventDisableTiming);
    }
    struct Job {
        int buf;
        uint64_t len;
    };
    std::mutex m;
    std::condition_variable cv;
    std::deque<Job> jobs;
    bool no_more = false, buf_free[2] = {true, true}, io_failed = false;
    cudaError_t copy_err = cudaSuccess;
    const int device = t->device;
    std::thread writer([&] {
        cudaSetDevice(device);
        for (;;) {
            Job j;
            {
                std::unique_lock<std::mutex> lk(m);
                cv.wait(lk, [&] { return no_more || !jobs.empty(); });
                if (jobs.empty()) return;
                j = jobs.front();
                jobs.pop_front();
            }
            const cudaError_t e = cudaEventSynchronize(copied[j.buf]);
            const bool ok = e == cudaSuccess && !io_failed && fwrite(w->h_slice[j.buf], 1, size_t(j.len), f) == size_t(j.len);
            {
                std::lock_guard<std::mutex> lk(m);
                if (e != cudaSuccess) copy_err = e;
                else if (!ok) io_failed = true;
                buf_free[j.buf] = true;
            }
            cv.notify_all();
        }
    });
    for (size_t i = 0; i < slices.size() && !rc; ++i) {
        const int b = int(i & 1);
        {
            std::unique_lock<std::mutex> lk(m);
            cv.wait(lk, [&] { return buf_free[b]; });
            if (io_failed || copy_err != cudaSuccess) break;
            buf_free[b] = false;
        }
        const Slice &sl = slices[i];
        rc = json_render_range(plan, sl.lo, sl.hi, pos[sl.lo], first_hit[sl.lo], first_hit[sl.hi], w->d_slice[b], w->s_comp);
        cudaError_t e = rc ? cudaSuccess : cudaEventRecord(rendered[b], w->s_comp);
        if (e == cudaSuccess && !rc) e = cudaStreamWaitEvent(w->s_copy, rendered[b], 0);
        if (e == cudaSuccess && !rc) e = cudaMemcpyAsync(w->h_slice[b], w->d_slice[b], sl.len, cudaMemcpyDeviceToHost, w->s_copy);
        if (e == cudaSuccess && !rc) e = cudaEventRecord(copied[b], w->s_copy);
        if (e != cudaSuccess) rc = cuda_fail(int(e), "svjg_filter_json_write: slice");
        if (rc) {
            std::lock_guard<std::mutex> lk(m);
            buf_free[b] = true;
            break;
        }
        {
            std::lock_guard<std::mutex> lk(m);
            jobs.push_back({b, sl.len});
        }
        cv.notify_all();
    }
    {
        std::lock_guard<std::mutex> lk(m);
        no_more = true;
    }
    cv.notify_all();
    writer.join();
    cudaStreamSynchronize(w->s_copy);
    json_plan_free(plan, w->s_comp);
    cudaStreamSynchronize(w->s_comp);
    for (int i = 0; i < 2; ++i) {
        cudaEventDestroy(rendered[i]);
        cudaEventDestroy(copied[i]);
    }
    const bool closed = fclose(f) == 0;
    if (!rc && copy_err != cudaSuccess) rc = cuda_fail(int(copy_err), "svjg_filter_json_write: copy");
    if (!rc && (io_failed || !closed)) rc = set_error(SVJG_E_IO, std::string("cannot write ") + path);
    if (rc) {
        remove(path);
        return rc;
    }
    if (json_len) *json_len = pos[num_sv] + 2;
    return SVJG_OK;
}

extern "C" int svjg_filter_json_host(svjg_tables *t, const uint8_t *gaf, uint64_t n_bytes, int64_t d_over, uint32_t *counts,
                                     svjg_filter_stats *stats, const char **json, uint64_t *json_len) {
    if (!json || !json_len) return set_error(SVJG_E_ARG, "svjg_filter_json_host: NULL argument");
    if (int rc = svjg_filter_json_begin(t, gaf, n_bytes, d_over, counts, stats)) return rc;
    return svjg_filter_json_finish(t, json, json_len);
}

// ---------------------------------------------------------------------------
// optional identity filter over the hit list (an extension, off by default)
// ---------------------------------------------------------------------------
// Aid of a stored line as filter-alignments.py:193-196 parses it: float() of what follows the LAST "id:f:" up to
// the next tab where the line holds that tag, else Am / Alen (columns 10 and 11).  The reference parses it and
// never uses it; its genotyper carries the gate commented out (predict-genotype.py:222).  false: float() raises.
static bool line_identity(const uint8_t *line, size_t len, double &out) {
    while (len && (line[len - 1] == ' ' || (line[len - 1] >= 9 && line[len - 1] <= 13) || (line[len - 1] >= 0x1c && line[len - 1] <= 0x1f)))
        --len;                                                        // line.rstrip() (:126)
    const uint8_t *tag = nullptr;
    for (size_t i = 0; i + 5 <= len; ++i)
        if (memcmp(line + i, "id:f:", 5) == 0) tag = line + i + 5;
    if (tag) {
        const uint8_t *e = tag;
        while (e < line + len && *e != '\t') ++e;
        std::string v(reinterpret_cast<const char *>(tag), size_t(e - tag));
        // float(): surrounding blanks, then a decimal literal, inf or nan; no hex, no underscores handled here
        size_t b = 0, n = v.size();
        while (b < n && (v[b] == ' ' || (v[b] >= 9 && v[b] <= 13))) ++b;
        while (n > b && (v[n - 1] == ' ' || (v[n - 1] >= 9 && v[n - 1] <= 13))) --n;
        v = v.substr(b, n - b);
        if (v.empty()) return false;
        for (char c : v)
            if (!(c >= '0' && c <= '9') && c != '.' && c != '+' && c != '-' && c != 'e' && c != 'E' && !strchr("infatyINFATY", c)) return false;
        if (v.find_first_of("xX") != std::string::npos) return false;
        char *end = nullptr;
        out = strtod(v.c_str(), &end);
        return end == v.c_str() + v.size();
    }
    // columns 10 and 11 (validated by the filter: digits only, Alen != 0)
    size_t col = 0, i = 0;
    uint64_t am = 0, alen = 0;
    for (; i < len && col < 11; ++i) {
        if (line[i] == '\t') {
            ++col;
            continue;
        }
        if (col == 9) am = am * 10 + uint64_t(line[i] - '0');
        else if (col == 10) alen = alen * 10 + uint64_t(line[i] - '0');
    }
    if (alen == 0) return false;
    out = double(am) / double(alen);
    return true;
}

extern "C" int svjg_hits_min_identity(const uint8_t *gaf, uint64_t n_bytes, uint32_t *hit_sv2, uint64_t *hit_off, uint32_t *hit_len,
                                      uint64_t *n_hits, double min_identity, uint32_t *counts, uint32_t num_sv) {
    if (!n_hits || (*n_hits && (!gaf || !hit_sv2 || !hit_off || !hit_len || !counts)))
        return set_error(SVJG_E_ARG, "svjg_hits_min_identity: NULL argument");
    uint64_t w = 0;
    for (uint64_t i = 0; i < *n_hits; ++i) {
        if (hit_off[i] + hit_len[i] > n_bytes || hit_sv2[i] >= 2ull * num_sv) return set_error(SVJG_E_ARG, "hit outside the GAF buffer");
        double id = 0;
        if (!line_identity(gaf + hit_off[i], hit_len[i], id)) {
            char msg[128];
            snprintf(msg, sizeof msg, "GAF line at byte %llu: the value of its id:f: tag is no number", (unsigned long long)hit_off[i]);
            return set_error(SVJG_E_INPUT, msg);
        }
        if (id >= min_identity) {
            hit_sv2[w] = hit_sv2[i];
            hit_off[w] = hit_off[i];
            hit_len[w] = hit_len[i];
            ++w;
        } else {
            --counts[hit_sv2[i]];
        }
    }
    *n_hits = w;
    return SVJG_OK;
}

// ---------------------------------------------------------------------------
// informative_aln.json   (json.dumps(d, sort_keys=True, indent=4))
// ---------------------------------------------------------------------------
namespace {

struct Out {                      // f == nullptr: everything stays in buf (a worker's share of the text)
    FILE *f;
    std::vector<char> buf;
    bool ok = true;
    explicit Out(FILE *fp) : f(fp) { buf.reserve(1 << 22); }
    void flush() {
        if (!f) return;
        if (!buf.empty() && fwrite(buf.data(), 1, buf.size(), f) != buf.size()) ok = false;
        buf.clear();
    }
    void put(const char *s, size_t n) {
        if (f && buf.size() + n > (1u << 22)) flush();
        buf.insert(buf.end(), s, s + n);
    }
    void put(const char *s) { put(s, strlen(s)); }
};

// JSON string with ensure_ascii=True; returns false on invalid UTF-8 (Python
// would have failed to decode the file)
bool put_json_string(Out &o, const uint8_t *s, size_t n) {
    static const char hex[] = "0123456789abcdef";
    char tmp[16];
    o.put("\"", 1);
    size_t run = 0;
    for (size_t i = 0; i < n;) {
        uint8_t c = s[i];
        if (c >= 0x20 && c < 0x80 && c != '"' && c != '\\') {
            ++run;
            ++i;
            continue;
        }
        if (run) o.put(reinterpret_cast<const char *>(s + i - run), run), run = 0;
        if (c < 0x80) {
            switch (c) {
                case '"': o.put("\\\"", 2); break;
                case '\\': o.put("\\\\", 2); break;
                case '\n': o.put("\\n", 2); break;
                case '\r': o.put("\\r", 2); break;
                case '\t': o.put("\\t", 2); break;
                case '\b': o.put("\\b", 2); break;
                case '\f': o.put("\\f", 2); break;
                default:
                    tmp[0] = '\\'; tmp[1] = 'u'; tmp[2] = '0'; tmp[3] = '0';
                    tmp[4] = hex[c >> 4]; tmp[5] = hex[c & 15];
                    o.put(tmp, 6);
            }
            ++i;
            continue;
        }
        uint32_t cp;
        int extra;
        if ((c & 0xE0) == 0xC0) cp = c & 0x1F, extra = 1;
        else if ((c & 0xF0) == 0xE0) cp = c & 0x0F, extra = 2;
        else if ((c & 0xF8) == 0xF0) cp = c & 0x07, extra = 3;
        else return false;
        if (i + size_t(extra) >= n) return false;
        for (int k = 1; k <= extra; ++k) {
            if ((s[i + k] & 0xC0) != 0x80) return false;
            cp = (cp << 6) | (s[i + k] & 0x3F);
        }
        if ((extra == 1 && cp < 0x80) || (extra == 2 && cp < 0x800) || (extra == 3 && cp < 0x10000) || cp > 0x10FFFF ||
            (cp >= 0xD800 && cp < 0xE000))
            return false;
        auto u4 = [&](uint32_t v) {
            tmp[0] = '\\'; tmp[1] = 'u';
            tmp[2] = hex[(v >> 12) & 15]; tmp[3] = hex[(v >> 8) & 15]; tmp[4] = hex[(v >> 4) & 15]; tmp[5] = hex[v & 15];
            o.put(tmp, 6);
        };
        if (cp >= 0x10000) {
            cp -= 0x10000;
            u4(0xD800 + (cp >> 10));
            u4(0xDC00 + (cp & 0x3FF));
        } else {
            u4(cp);
        }
        i += size_t(extra) + 1;
    }
    if (run) o.put(reinterpret_cast<const char *>(s + n - run), run);
    o.put("\"", 1);
    return true;
}

}  // namespace

// out_path: the file to write; or mem: the text is appended there instead
static int emit_json(const svjg_tables *t, const uint8_t *gaf, uint64_t n_bytes, const uint32_t *hit_sv2, const uint64_t *hit_off,
                     const uint32_t *hit_len, uint64_t n_hits, const char *out_path, std::vector<char> *mem) {
    if (!t || (!out_path && !mem) || (n_hits && (!gaf || !hit_sv2 || !hit_off || !hit_len)))
        return set_error(SVJG_E_ARG, "svjg_emit_informative_json: NULL argument");
    const uint64_t n2 = uint64_t(t->sv_ids.size()) * 2;
    // counting sort by (sv, allele); inside a list the reference appends in file order
    std::vector<uint64_t> start(n2 + 1, 0);
    for (uint64_t i = 0; i < n_hits; ++i) {
        if (hit_sv2[i] >= n2) return set_error(SVJG_E_ARG, "hit with an sv index outside the tables");
        if (hit_off[i] + hit_len[i] > n_bytes) return set_error(SVJG_E_ARG, "hit outside the GAF buffer");
        ++start[hit_sv2[i] + 1];
    }
    for (uint64_t k = 0; k < n2; ++k) start[k + 1] += start[k];
    std::vector<uint64_t> order(n_hits);
    {
        std::vector<uint64_t> cur(start.begin(), start.end() - 1);
        for (uint64_t i = 0; i < n_hits; ++i) order[cur[hit_sv2[i]]++] = i;
    }
    for (uint64_t k = 0; k < n2; ++k)
        std::sort(order.begin() + start[k], order.begin() + start[k + 1],
                  [&](uint64_t x, uint64_t y) { return hit_off[x] < hit_off[y]; });

    FILE *f = mem ? nullptr : fopen(out_path, "wb");
    if (!mem && !f) return set_error(SVJG_E_IO, std::string("cannot write ") + out_path);
    auto sink = [&](const char *p, size_t n) {
        if (mem) {
            mem->insert(mem->end(), p, p + n);
            return true;
        }
        return fwrite(p, 1, n, f) == n;
    };
    // The text of a key does not depend on the others: keys are rendered by several threads, a batch
    // (about 256 MB of lines) at a time, every thread a run of keys with about the same number of
    // bytes, and written in key order.  Every key starts with ",\n    "; the first one of the file has
    // its comma turned into the opening brace (same length).
    auto render = [&](uint64_t sv_lo, uint64_t sv_hi, Out &o, bool &utf8_ok) {
        for (uint64_t sv = sv_lo; sv < sv_hi && utf8_ok; ++sv) {
            if (start[2 * sv] == start[2 * sv + 2]) continue;   // a key exists only once something was appended (:163)
            o.put(",\n    ");
            const std::string &id = t->sv_ids[sv];
            utf8_ok &= put_json_string(o, reinterpret_cast<const uint8_t *>(id.data()), id.size());
            o.put(": [\n        ");
            for (int al = 0; al < 2 && utf8_ok; ++al) {
                uint64_t b = start[2 * sv + al], e = start[2 * sv + al + 1];
                if (b == e) {
                    o.put("[]");
                } else {
                    o.put("[\n            ");
                    for (uint64_t k = b; k < e && utf8_ok; ++k) {
                        uint64_t i = order[k];
                        const uint8_t *line = gaf + hit_off[i];
                        size_t len = hit_len[i];
                        const void *cgz = memmem(line, len, "cg:Z:", 5);      // line.split("cg:Z:")[0]  (:166)
                        if (cgz) len = size_t(static_cast<const uint8_t *>(cgz) - line);
                        if (k != b) o.put(",\n            ");
                        utf8_ok &= put_json_string(o, line, len);
                    }
                    o.put("\n        ]");
                }
                if (al == 0) o.put(",\n        ");
            }
            o.put("\n    ]");
        }
    };
    const uint64_t n_sv = n2 / 2;
    std::vector<uint64_t> weight(n_sv + 1, 0);                  // bytes of lines up to key sv (prefix sums)
    for (uint64_t sv = 0; sv < n_sv; ++sv) {
        uint64_t w = 0;
        for (uint64_t k = start[2 * sv]; k < start[2 * sv + 2]; ++k) w += hit_len[order[k]] + 16;
        weight[sv + 1] = weight[sv] + w;
    }
    unsigned n_thr = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    if (weight[n_sv] < (8u << 20)) n_thr = 1;
    uint64_t batch_bytes = 256ull << 20;
    if (const char *e = getenv("SVJG_JSON_THREADS")) n_thr = unsigned(std::max(1, std::min(64, atoi(e))));   // test hooks
    if (const char *e = getenv("SVJG_JSON_BATCH")) batch_bytes = uint64_t(std::max(1, atoi(e)));
    bool any = false, utf8_ok = true, io_ok = true;
    for (uint64_t lo = 0; lo < n_sv && utf8_ok && io_ok;) {
        uint64_t hi = std::upper_bound(weight.begin() + lo, weight.end(), weight[lo] + batch_bytes) - weight.begin();
        hi = std::min<uint64_t>(std::max<uint64_t>(hi, lo + 1), n_sv);
        std::vector<uint64_t> cutv(n_thr + 1, lo);
        for (unsigned p = 1; p < n_thr; ++p) {
            const uint64_t target = weight[lo] + (weight[hi] - weight[lo]) * p / n_thr;
            cutv[p] = std::min<uint64_t>(hi, std::lower_bound(weight.begin() + lo, weight.begin() + hi, target) - weight.begin());
        }
        cutv[n_thr] = hi;
        for (unsigned p = 1; p <= n_thr; ++p) cutv[p] = std::max(cutv[p], cutv[p - 1]);
        std::vector<Out> outs;
        outs.reserve(n_thr);
        for (unsigned p = 0; p < n_thr; ++p) outs.emplace_back(nullptr);
        std::vector<char> okv(n_thr, 1);
        std::vector<std::thread> pool;
        for (unsigned p = 1; p < n_thr; ++p)
            pool.emplace_back([&, p]() {
                bool u = true;
                render(cutv[p], cutv[p + 1], outs[p], u);
                okv[p] = u;
            });
        {
            bool u = true;
            render(cutv[0], cutv[1], outs[0], u);
            okv[0] = u;
        }
        for (auto &th : pool) th.join();
        for (unsigned p = 0; p < n_thr && io_ok; ++p) {
            utf8_ok &= okv[p] != 0;
            std::vector<char> &b = outs[p].buf;
            if (b.empty()) continue;
            if (!any) b[0] = '{';
            any = true;
            io_ok = sink(b.data(), b.size());
        }
        lo = hi;
    }
    if (io_ok) io_ok = any ? sink("\n}", 2) : sink("{}", 2);
    bool ok = (f ? fclose(f) == 0 : true) && io_ok;
    if (!utf8_ok) return set_error(SVJG_E_INPUT, "GAF text is not valid UTF-8 (the reference cannot read it)");
    if (!ok) return set_error(SVJG_E_IO, std::string("write failed: ") + (out_path ? out_path : "(memory)"));
    return SVJG_OK;
}

extern "C" int svjg_emit_informative_json(const svjg_tables *t, const uint8_t *gaf, uint64_t n_bytes,
                                          const uint32_t *hit_sv2, const uint64_t *hit_off, const uint32_t *hit_len,
                                          uint64_t n_hits, const char *out_path) {
    if (!out_path) return set_error(SVJG_E_ARG, "svjg_emit_informative_json: NULL argument");
    return emit_json(t, gaf, n_bytes, hit_sv2, hit_off, hit_len, n_hits, out_path, nullptr);
}

// the same text in memory: *out is released with svjg_buffer_free
extern "C" int svjg_emit_informative_json_mem(const svjg_tables *t, const uint8_t *gaf, uint64_t n_bytes,
                                              const uint32_t *hit_sv2, const uint64_t *hit_off, const uint32_t *hit_len,
                                              uint64_t n_hits, char **out, uint64_t *out_len) {
    if (!out || !out_len) return set_error(SVJG_E_ARG, "svjg_emit_informative_json_mem: NULL argument");
    std::vector<char> mem;
    const int rc = emit_json(t, gaf, n_bytes, hit_sv2, hit_off, hit_len, n_hits, nullptr, &mem);
    if (rc) return rc;
    char *p = static_cast<char *>(malloc(mem.size() ? mem.size() : 1));
    if (!p) return set_error(SVJG_E_NOMEM, "out of memory");
    memcpy(p, mem.data(), mem.size());
    *out = p;
    *out_len = mem.size();
    return SVJG_OK;
}
