// Internal declarations shared by the translation units of libsvjg.so.
#pragma once
#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "../../include/svjg.h"
#include "svjg_common.h"

namespace svjg {
struct HostWs;
struct JsonKeys;
struct JsonPlan;
}

struct svjg_tables {
    std::vector<std::string> sv_ids;          // byte-sorted distinct sv ids
    std::vector<svjg::LinkSlot> links;
    std::vector<svjg::NodeSlot> nodes;
    std::vector<svjg::PNodeSlot> pnodes;
    std::vector<uint8_t> blob;
    std::vector<uint32_t> entries;
    uint32_t n_keys = 0, n_link_slots = 0, n_alt = 0, n_nodes = 0;
    uint32_t filter_flags = 0;                // SVJG_FLAG_* passed to the filter kernel
    // device image
    int device = -1;
    void *d_links = nullptr, *d_nodes = nullptr, *d_blob = nullptr, *d_entries = nullptr, *d_pnodes = nullptr;
    svjg::DevTables dev{};
    // lazily created workspace of svjg_filter_host
    svjg::HostWs *ws = nullptr;
    // lazily created device copy of the sv ids as JSON strings (json.cu)
    svjg::JsonKeys *json_keys = nullptr;
};

// counters of S samples against one catalogue (api.cu), genotyped block by block (genotype.cu)
struct svjg_cohort {
    svjg_tables *t = nullptr;
    uint32_t n_samples = 0, num_sv = 0;
    uint32_t *d_counts = nullptr;             // [n_samples][num_sv][2], sample-major
    cudaStream_t stream = nullptr;
    std::vector<double> lut;                  // host copy of what d_lut holds
    double *d_lut = nullptr;
    uint8_t *d_blk = nullptr;                 // inputs and results of the last block
    size_t blk_cap = 0;
    uint32_t blk_n = 0;                       // records of the last block genotyped (0: none)
    size_t blk_gt = 0;                        // offset of its gt codes [blk_n][n_samples] in d_blk
    size_t blk_pl = 0, blk_fl = 0;            // offsets of its pl [blk_n][n_samples][3] and flags [blk_n][n_samples]
    size_t blk_ty = 0;                        // offset of its svtype codes [blk_n]
    bool blk_qc = false;                      // svjg_cohort_qc_add has packed the last block
    uint32_t *d_qc = nullptr;                 // svjg_cohort_qc_begin: histogram [n_samples][5][8], then (qc_pairs) the
                                              // bit planes C, H, A [3][n_samples][qc_stride]
    uint32_t qc_words = 0, qc_used = 0;       // words of a plane row the caller announced, and packed so far
    size_t qc_stride = 0;                     // qc_words rounded up to whole K slabs of the pair kernel
    bool qc_on = false, qc_pairs = false;
    uint8_t *d_site = nullptr;                // site statistics of the last block (svjg_cohort_site_stats)
    size_t site_cap = 0;
    std::vector<double> plw;                  // host copy of what d_plw holds: T[k] = 10^(-k/10) (svjg_cohort_posteriors)
    double *d_plw = nullptr;
    uint8_t *d_post = nullptr;                // inputs and results of the last svjg_cohort_posteriors call
    size_t post_cap = 0;
    uint8_t *d_ploidy = nullptr;              // svjg_cohort_set_ploidy: table [n_classes][n_sexes], then sex [n_samples]
    uint32_t n_classes = 0, n_sexes = 0;
};

namespace svjg {
// where the bytes of a file lie on the device(s): range k = file offsets [start[k], start[k + 1]) at base[k]
// (device 0's own memory or a peer's, read over NVLink).  One range for a file resident on one device.
constexpr int MAX_RANGES = 8;
struct LineSrc {
    const uint8_t *base[MAX_RANGES];
    uint64_t start[MAX_RANGES];
    uint32_t n;
};
int set_error(int code, const std::string &msg);
int cuda_fail(int cuda_err, const char *what);   // records the message, returns SVJG_E_CUDA
void free_host_ws(svjg_tables *t);
void free_json_keys(svjg_tables *t);
// informative_aln.json rendered on the device from hits in device memory (json.cu); *d_out is released with cudaFreeAsync
int json_render_device(svjg_tables *t, const LineSrc &src, const uint32_t *d_hit_sv2, const uint64_t *d_hit_off,
                       const uint32_t *d_hit_len, uint64_t n_hits, const uint32_t *d_counts, uint8_t **d_out, uint64_t *out_len,
                       cudaStream_t st);
// the same in steps, for a text that leaves the device slice by slice (json.cu; see there)
int json_plan(svjg_tables *t, const LineSrc &src, const uint32_t *d_hit_sv2, const uint64_t *d_hit_off, const uint32_t *d_hit_len,
              uint64_t n_hits, const uint32_t *d_counts, JsonPlan **out_plan, cudaStream_t st);
uint64_t json_plan_bytes(const JsonPlan *plan);
uint32_t json_plan_keys(const JsonPlan *plan);
int json_plan_key_positions(const JsonPlan *plan, uint64_t *pos, uint64_t *first_hit, cudaStream_t st);
int json_render_range(const JsonPlan *plan, uint32_t sv_lo, uint32_t sv_hi, uint64_t base, uint64_t h_lo, uint64_t h_hi, uint8_t *d_out,
                      cudaStream_t st);
void json_plan_free(JsonPlan *plan, cudaStream_t st);
// svjg_filter_device with absolute 64-bit hit offsets (d_hit_off64 != NULL); filter.cu
int filter_device_abs(const svjg_tables *t, const uint8_t *d_gaf, uint64_t n_bytes, uint64_t base_offset, int64_t d_over,
                      uint32_t *d_counts, uint32_t *d_hit_sv2, uint32_t *d_hit_off, uint64_t *d_hit_off64, uint32_t *d_hit_len,
                      uint64_t hit_cap, svjg_filter_stats *d_stats, void *stream, bool inside_buffer = false);
}  // namespace svjg

#define SVJG_CUDA(call)                                                        \
    do {                                                                       \
        cudaError_t _e = (call);                                               \
        if (_e != cudaSuccess) return svjg::cuda_fail(int(_e), #call);        \
    } while (0)
