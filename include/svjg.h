/* svjg.h — C ABI of libsvjg.so: the B200-native post-mapping hot path of
 * SVJedi-graph (informative-alignment filter + per-SV allele counts + genotype
 * likelihoods).
 *
 * The reference has no in-process plugin API: its boundary is two CLI stages
 * glued by files (svjedi-graph.py:113-128).  Each entry point below cites the
 * reference code it replaces (paths relative to the reference checkout).
 * Plain pointers and sizes only; no torch types.  Pointers named d_* are CUDA
 * device pointers owned by the caller; everything else is host memory.
 *
 * Every function returns 0 (SVJG_OK) or a non-zero SVJG_E_* code; a drop-in
 * front-end turns any non-zero code into process exit status 1, which is what
 * the reference's uncaught Python exceptions produce (svjedi-graph.py:117,127).
 * svjg_last_error() gives a human-readable message for the calling thread.
 */
#ifndef SVJG_H
#define SVJG_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SVJG_OK 0
#define SVJG_E_CUDA 1          /* CUDA runtime failure                                */
#define SVJG_E_ARG 2           /* bad argument (NULL, misaligned, too large)          */
#define SVJG_E_IO 3            /* file could not be read / written                    */
#define SVJG_E_JSON 4          /* <prefix>_svs_edges.json is not the expected JSON    */
#define SVJG_E_INPUT 5         /* input on which the reference raises (exit status 1) */
#define SVJG_E_HITS_OVERFLOW 6 /* hit buffers too small: re-run with >= n_hits slots  */
#define SVJG_E_NOMEM 7
#define SVJG_E_UNSUPPORTED 8   /* a spelling this library does not reproduce (see svjg_vcf_parse)  */

/* reason codes stored in svjg_filter_stats.status when a GAF line would make the
 * reference raise (SURVEY.md appendix A.4) */
#define SVJG_BAD_COLUMNS 1   /* blank line / fewer than 12 columns  (filter-alignments.py:185-187) */
#define SVJG_BAD_INT 2       /* non-integer numeric column          (:189-191)                     */
#define SVJG_BAD_ALEN 3      /* Alen == 0 and no id:f: tag          (:196)                         */
#define SVJG_BAD_PATH 4      /* empty path, or token with nothing in front of it (:206, :366)      */
#define SVJG_BAD_ALTNODE 5   /* alt node of a hit record missing from the GFA (:346)               */
#define SVJG_BAD_NODENAME 6  /* reference-node name without start-end (:342, :349)                 */
#define SVJG_BAD_ENTRY 7     /* sv id without ':' or allele not 0/1 in svs_edges (:160, :166)      */
#define SVJG_BAD_SHORTLINE 8 /* a line shorter than 16 bytes (cannot hold 12 columns)              */
#define SVJG_BAD_RANGE 9     /* integer beyond 18 digits (unsupported; the reference has bigints)  */

typedef struct svjg_tables svjg_tables;

const char *svjg_version(void);
const char *svjg_last_error(void);

/* ---- graph tables --------------------------------------------------------
 * Replaces filter-alignments.py:95-98 (json.load of <prefix>_svs_edges.json into
 * d_link_sv) and :103-113 (alt-node length scan of the GFA).  Builds, on the
 * host, a hash of link key -> [(sv index, allele)] and a hash of alt-node name
 * -> sequence length; sv indices are ranks in the byte-sorted list of distinct
 * sv ids (the order json.dumps(sort_keys=True) prints them, :175). */
int svjg_tables_load(const char *svs_edges_json_path, const char *gfa_path, svjg_tables **out);
int svjg_tables_from_memory(const char *edges_json, size_t edges_len, const char *gfa, size_t gfa_len,
                            svjg_tables **out);
void svjg_tables_free(svjg_tables *t);
uint32_t svjg_tables_num_sv(const svjg_tables *t);
uint32_t svjg_tables_num_links(const svjg_tables *t);     /* distinct link keys        */
uint32_t svjg_tables_num_alt_nodes(const svjg_tables *t);
uint64_t svjg_tables_device_bytes(const svjg_tables *t);  /* size of the device image  */
/* alt_node_len[name] of filter-alignments.py:103-113 as the kernels will find it (the same hash
 * probes, on the host copy of the tables): the sequence length, -1 when the GFA gave the name no
 * length, -2 if the two node tables of the image disagree (never, short of a bug).  The GFA is read
 * as the reference reads it: text mode ("\n", "\r\n" and a lone "\r" end a line), an 'S' line
 * whose name has a '.' after its last ':' is an alt node, its length is len() of the third column
 * of the right-stripped line; a damaged 'S' line the reference raises on is SVJG_E_INPUT. */
int64_t svjg_tables_alt_node_len(const svjg_tables *t, const char *name, uint32_t len);
/* FNV-1a over the whole host image (hash tables, name blob, entries, sv ids, flags): two handles with
 * the same value upload the same bytes (regression hook for the table builder) */
uint64_t svjg_tables_image_hash(const svjg_tables *t);
/* sv id string of index i (not NUL terminated); NULL when i is out of range */
const char *svjg_tables_sv_id(const svjg_tables *t, uint32_t i, uint32_t *len);
/* index of an sv id, or UINT32_MAX — what `in_sv in dict` needs (predict-genotype.py:216) */
uint32_t svjg_tables_find_sv(const svjg_tables *t, const char *sv_id, uint32_t len);
/* Filter behaviour switches (OR-ed in; EXACT_CHECKS is set automatically when svs_edges
 * holds an entry the reference would raise on):
 *   SVJG_FLAG_EXACT_CHECKS  probe the link table even for links whose breakpoint-overlap
 *                           test fails, so stats.n_checks counts every evaluation the
 *                           reference makes (needed to mirror the -O crash, :269)
 *   SVJG_FLAG_FORCE_GENERAL send every multi-node line through the general routine
 *                           (test hook: fast path and general routine must agree) */
#define SVJG_FLAG_EXACT_CHECKS 1u
#define SVJG_FLAG_FORCE_GENERAL 2u
int svjg_tables_set_flags(svjg_tables *t, uint32_t flags);
/* a second handle with the same host image and no device image: several GPUs of a node get one handle each */
int svjg_tables_clone(const svjg_tables *t, svjg_tables **out);
/* copies the device image to `device` (cudaMalloc inside; freed by svjg_tables_free) */
int svjg_tables_to_device(svjg_tables *t, int device);

/* ---- filter + count (kernels 1-3) ------------------------------------------
 * Replaces the whole per-line loop filter-alignments.py:123-166: line split and
 * integer parse (read_gaf_line :184-198), path tokenising (extract_nodes
 * :351-373), strands and links (get_aln_links :200-219), forward / reverse key
 * probes (:141-148), the breakpoint-overlap test (check_bkpt_overlap :258-273,
 * get_node_len :343-349) and the append (:160-166), which becomes
 *   d_counts[2*sv + allele] += 1          (what predict-genotype.py:219-226 counts)
 *   hit (2*sv + allele, line offset, line length)   appended at an atomic cursor.
 * The text the reference stores per hit (:166) is gaf[off : off+len] cut at the
 * first "cg:Z:" — svjg_emit_informative_json() does that cut when it prints.
 *
 * d_gaf must be 16-byte aligned; n_bytes < 2^32 (shard larger files by lines).
 * d_counts (2*num_sv u32) and d_stats are ACCUMULATED, so several shards can be
 * filtered into one set of counters: clear them first with svjg_filter_reset().
 * Asynchronous on `stream` (a cudaStream_t); nothing is read back. */
typedef struct svjg_filter_stats {
    uint64_t n_hits;     /* hits produced; > hit_cap means the tail was dropped  */
    uint64_t n_records;  /* GAF lines seen                                       */
    uint64_t n_multi;    /* lines whose path has >= 2 nodes (:133)               */
    uint64_t n_checks;   /* overlap tests evaluated (-O given => reference raises if > 0, :269) */
    uint64_t status;     /* 0, or the first SVJG_BAD_* reason                    */
    uint64_t err_offset; /* byte offset of the lowest offending line             */
    uint64_t n_generic;  /* records that took the general (quirk-exact) path     */
    uint64_t n_exact;      /* lines the exact kernel took (irregular shape, too long for the window) */
} svjg_filter_stats;

int svjg_filter_reset(uint32_t *d_counts, uint32_t num_sv, svjg_filter_stats *d_stats, void *stream);
int svjg_filter_device(const svjg_tables *t, const uint8_t *d_gaf, uint64_t n_bytes, uint64_t base_offset,
                       int64_t d_over, uint32_t *d_counts, uint32_t *d_hit_sv2, uint32_t *d_hit_off,
                       uint32_t *d_hit_len, uint64_t hit_cap, svjg_filter_stats *d_stats, void *stream);

/* Text-mode line ends as the reference's `open(gaf)` gives them (filter-alignments.py:123): "\r\n" and a lone
 * "\r" become "\n", in place, one pass; returns the new length.  A front-end calls it before the filter when
 * its bytes may hold carriage returns (the kernels split at "\n" only). */
uint64_t svjg_translate_newlines(uint8_t *p, uint64_t n);

/* Measurement and test aids of the filter (no reference analogue; process-wide, not thread-safe against
 * running filter calls).
 *   svjg_filter_profile(1)   every later svjg_filter_device call records CUDA events around its scan
 *                            kernel on the caller's stream; svjg_filter_scan_ms() waits for the last such
 *                            call on the current device and returns that kernel's duration
 *   svjg_filter_tune(knob, value)   value 0 restores the default
 *     SVJG_TUNE_TILE_BYTES   bytes of the shard a warp owns per step, instead of the probe kernel's choice
 *     SVJG_TUNE_TILE_LINES   lines a tile should hold (the probe kernel's target; default 30)
 *     SVJG_TUNE_SCAN_BLOCKS  blocks per SM the scan kernel is sized for (6 or 8): trades window size for warps
 *     SVJG_TUNE_SCAN_ONLY    1: the scan kernel stops behind its byte-class phase, nothing else runs
 *     SVJG_TUNE_POOL_UNITS   16-byte units of the exact kernel's bump pool (forces its no-room fallbacks) */
#define SVJG_TUNE_TILE_BYTES 1
#define SVJG_TUNE_TILE_LINES 2
#define SVJG_TUNE_SCAN_BLOCKS 3
#define SVJG_TUNE_SCAN_ONLY 4
#define SVJG_TUNE_POOL_UNITS 5
int svjg_filter_tune(int knob, int value);
int svjg_filter_profile(int enable);
int svjg_filter_scan_ms(float *ms);

/* Lines end at '\n'.  The reference opens the GAF in text mode, where "\r\n" and a lone "\r" end a
 * line as well (and are stored as "\n"): a caller whose bytes may contain carriage returns translates
 * them first, as the drop-in front-ends do (svjg/alnfilter.py: translate_newlines).
 *
 * Same, from HOST memory: stages the bytes to the device in pinned chunks cut at
 * line ends, overlapping copies with the kernel; returns counts, stats and the
 * hits (offsets are absolute in `gaf`) in host arrays.  `hit_*` may be NULL to
 * skip the hit list (counts only).  Synchronous.  Returns SVJG_E_INPUT with
 * stats->status set where the reference would raise. */
int svjg_filter_host(svjg_tables *t, const uint8_t *gaf, uint64_t n_bytes, int64_t d_over, uint32_t *counts,
                     uint32_t *hit_sv2, uint64_t *hit_off, uint32_t *hit_len, uint64_t hit_cap,
                     svjg_filter_stats *stats);

/* The same, with `informative_aln.json` (filter-alignments.py:160-175) rendered ON THE DEVICE: the file stays
 * resident in device memory while it is filtered, the hit tuples never leave the device; they are put into
 * list order there (by sv id and allele, then file order, :166), the escaped text is assembled in device
 * memory and crosses PCIe once, as text.  *json points into a page-locked buffer owned by `t`, valid until the
 * next call with `t` or svjg_tables_free.  SVJG_E_UNSUPPORTED: the device renderer declines (a non-ASCII byte
 * in a stored line, a list beyond 64 Ki entries, a file that does not fit device memory beside its hits and its
 * text) -- use svjg_filter_host + svjg_emit_informative_json; nothing is lost, those stream the file in chunks. */
int svjg_filter_json_host(svjg_tables *t, const uint8_t *gaf, uint64_t n_bytes, int64_t d_over, uint32_t *counts,
                          svjg_filter_stats *stats, const char **json, uint64_t *json_len);
/* The same in two halves, for a caller that genotypes (which needs the counters only) while the text is rendered
 * and copied: _begin returns once counters and stats are on the host; _finish renders the text and waits for it.
 * Both may be called from different threads, one after the other. */
int svjg_filter_json_begin(svjg_tables *t, const uint8_t *gaf, uint64_t n_bytes, int64_t d_over, uint32_t *counts,
                           svjg_filter_stats *stats);
int svjg_filter_json_finish(svjg_tables *t, const char **json, uint64_t *json_len);
/* One file on several devices: range k of the file (cut at line ends, in file order) goes through
 * svjg_filter_json_begin_at with the tables on device k -- `gaf` points at the range, `base` is its offset in the
 * file, hits carry file offsets; one host thread per device.  svjg_filter_json_gather then copies the hit tuples of
 * devices 1.. to device 0 (peer copies), uploads the counters the caller has summed, and lets ts[0]'s
 * svjg_filter_json_finish / _write render the whole text, reading every line where it lies: device 0's memory or a
 * peer's over NVLink.  At most 8 ranges.  SVJG_E_UNSUPPORTED: no peer access between the devices. */
int svjg_filter_json_begin_at(svjg_tables *t, const uint8_t *gaf, uint64_t n_bytes, uint64_t base, int64_t d_over,
                              uint32_t *counts, svjg_filter_stats *stats);
int svjg_filter_json_gather(svjg_tables **ts, int n, const uint32_t *counts_sum);
/* The second half for a text that goes to a file (the `with open(...)` of filter-alignments.py:174-175): whole keys
 * are rendered slice by slice (about `slice_bytes` each, 0 = 64 MiB), copied into one of two page-locked slices and
 * written by a thread of its own while the next slice is rendered and copied; neither the device nor the host hold
 * the whole text.  *json_len (may be NULL) = bytes written.  Declines like svjg_filter_json_finish (nothing is
 * written then); a file that cannot be written: SVJG_E_IO, and what was written of it is removed. */
int svjg_filter_json_write(svjg_tables *t, const char *path, uint64_t slice_bytes, uint64_t *json_len);

/* Optional identity filter (an extension, off by default; the reference parses the identity of every alignment,
 * filter-alignments.py:193-196, and never uses it; predict-genotype.py:222 carries the gate commented out):
 * drops from a HOST hit list the hits whose line has Aid < min_identity -- Aid as :193-196 defines it, float() of
 * the text behind the last "id:f:" up to the next tab, else Am / Alen -- compacting the three arrays in place and
 * taking the dropped hits off the counters.  SVJG_E_INPUT where float() would raise. */
int svjg_hits_min_identity(const uint8_t *gaf, uint64_t n_bytes, uint32_t *hit_sv2, uint64_t *hit_off, uint32_t *hit_len,
                           uint64_t *n_hits, double min_identity, uint32_t *counts, uint32_t num_sv);

/* ---- genotype (kernel 4) ----------------------------------------------------
 * Replaces likelihood() / allele_normalization() / encode_genotype()
 * (predict-genotype.py:281-346) and the gate at :216 for n SVs of a VCF.
 *   sv_index[i]  index into d_counts pairs, or UINT32_MAX if the key is not in the tables
 *   svtype[i]    0 DEL, 1 INS, 2 INV, 3 BND, 255 other;  bit 7 set = |length| < 50 (:216);
 *                bit 6 set = the key is present even if both counts are 0 (a hand-made JSON;
 *                with counters that come from the filter a key exists iff it has a hit)
 *   log10_1me, log10_e, log10_half : math.log10(1-e), math.log10(e), math.log10(1/2)
 *                as computed by the caller's libm (the reference uses CPython's)
 *   lut          log10(C(n,k)) at [n*(n+1)/2 + k] for 0 <= k <= n <= lut_nmax, bit-equal
 *                to CPython's math.log10(math.comb(n,k)) (:313); SVs whose rounded
 *                counts exceed lut_nmax get flag SVJG_GT_NEED_K and are re-run with
 *                k_override[i] (NaN = not given; pointer may be NULL)
 * Outputs per SV: pl[3] = int(-10*(lik+comb)) exact (:319-323); gt 0,1,2 = 0/0,0/1,1/1,
 * 3 = ./. ; ad2[2] = normalised counts in HALF units (:327-338); flags below. */
#define SVJG_GT_GENOTYPED 1 /* passed the gate at predict-genotype.py:216 */
#define SVJG_GT_HALVED_0 2  /* c1 was normalised (prints as float)        */
#define SVJG_GT_HALVED_1 4  /* c2 was normalised                          */
#define SVJG_GT_NEED_K 8    /* log10 C(n,k) not available: pl invalid     */

int svjg_genotype_device(const uint32_t *d_counts, const uint32_t *d_sv_index, const uint8_t *d_svtype,
                         uint32_t n, int64_t min_support, double log10_1me, double log10_e,
                         double log10_half, const double *d_lut, uint32_t lut_nmax,
                         const double *d_k_override, int64_t *d_pl, uint8_t *d_gt, uint32_t *d_ad2,
                         uint8_t *d_flags, void *stream);

/* The same from HOST arrays (counts [num_counts][2]); device buffers are the call's own.  Synchronous. */
int svjg_genotype_host(const uint32_t *counts, uint32_t num_counts, const uint32_t *sv_index, const uint8_t *svtype,
                       uint32_t n, int64_t min_support, double log10_1me, double log10_e, double log10_half,
                       const double *lut, uint32_t lut_nmax, const double *k_override, int64_t *pl, uint8_t *gt,
                       uint32_t *ad2, uint8_t *flags);

/* ---- cohorts: one catalogue genotyped in many samples -------------------------
 * The reference genotypes one sample per run; a cohort of S samples keeps the counters of every sample on the
 * device at once, so the tables are loaded and the context created once.  The counter matrix is [S][num_sv][2]
 * u32 (sample-major: each sample's slice is the counter array of svjg_filter_host).
 *   svjg_cohort_create      a zeroed counter matrix on the device of `t` (t must stay alive and on its device)
 *   svjg_cohort_filter      svjg_filter_host into sample `sample`'s counters, from host bytes: ACCUMULATED (several
 *                           files of one sample are counted together, as the reference counts the GAFs it appends
 *                           into one file); no hit list.  Synchronous.  SVJG_E_INPUT with stats->status and
 *                           stats->err_offset (offset within `gaf`) where the reference would raise
 *   svjg_cohort_read_counts / svjg_cohort_load_counts   host copy [num_sv][2] of one sample's counters, out / in
 *   svjg_cohort_genotype    svjg_genotype_host for n records in every sample (no k_override: cells whose rounded
 *                           counts exceed lut_nmax get SVJG_GT_NEED_K; the caller recomputes those cells from their
 *                           counters, e.g. with svjg_genotype_host).  Outputs are host arrays [n][S]: pl [n][S][3],
 *                           gt, flags [n][S], ad2 [n][S][2].  The LUT and the block buffers are cached in the handle.
 *                           Synchronous.
 *   svjg_cohort_site_stats  population statistics of the records of the last svjg_cohort_genotype call (n must be
 *                           its record count), from the gt codes that call left on the device; only these 32 B per
 *                           record come back.  gcount [n][4] u32 = (r0, h, r2, m): cells with 0/0, 0/1, 1/1 and the
 *                           rest (./.).  hwe [n], exchet [n]: the HWE exact test and the excess-heterozygosity p of
 *                           (r0, h, r2) (Wigginton, Cutler & Abecasis 2005, in the fixed double-precision form of
 *                           DESIGN.md §8a; 1 and 1 when no allele is rare, NS = 0 included).  SVJG_E_ARG when
 *                           4 (S + 1)^2 >= 2^53.  The gt codes on the device are final: the NEED_K cells a caller
 *                           recomputes keep their genotype.  Synchronous. */
typedef struct svjg_cohort svjg_cohort;
int svjg_cohort_create(svjg_tables *t, uint32_t n_samples, svjg_cohort **out);
void svjg_cohort_free(svjg_cohort *c);
int svjg_cohort_filter(svjg_cohort *c, uint32_t sample, const uint8_t *gaf, uint64_t n_bytes, int64_t d_over,
                       svjg_filter_stats *stats);
int svjg_cohort_read_counts(svjg_cohort *c, uint32_t sample, uint32_t *counts);
int svjg_cohort_load_counts(svjg_cohort *c, uint32_t sample, const uint32_t *counts);
int svjg_cohort_genotype(svjg_cohort *c, const uint32_t *sv_index, const uint8_t *svtype, uint32_t n, int64_t min_support,
                         double log10_1me, double log10_e, double log10_half, const double *lut, uint32_t lut_nmax,
                         int64_t *pl, uint8_t *gt, uint32_t *ad2, uint8_t *flags);
int svjg_cohort_site_stats(svjg_cohort *c, uint32_t n, uint32_t *gcount, double *hwe, double *exchet);

/* Page-locked host memory (cudaHostAlloc) for file buffers and results: copies to and from it run
 * at PCIe speed.  For callers that do not want a tensor library just to pin memory. */
int svjg_host_alloc(uint64_t bytes, void **out);
int svjg_host_free(void *p);
/* page-lock / release memory the caller owns; create the CUDA context of a device (about a second:
 * a front-end calls it from a thread while it reads its input files) */
int svjg_host_register(void *p, uint64_t bytes);
int svjg_host_unregister(void *p);
int svjg_device_init(int device);

/* ---- counters of several GPUs (one process per GPU, one node) ----------------
 * The reference has no analogue (single process).  GAF records shard by read, so every rank
 * filters its shard into its own counters; predict-genotype.py:219-226 needs their sum.
 * Instead of an all-reduce followed by the genotype kernel, every rank keeps its counters in an
 * exchange region that the other ranks map (CUDA IPC over NVLink peer access), and the genotype
 * kernel of a rank sums, for its SVs only, the counters of all ranks where they lie.
 *   region = 64 flag words, then three counter buffers [num_sv][2] u32 taken in turn by the steps (buffer
 *   `parity` = step % 3): a rank may filter step k + 1 -- on another stream even while its own genotype kernel of
 *   step k still waits for the slowest rank -- while peers read step k; buffer k % 3 is written again by step
 *   k + 3, which the caller starts behind its genotype kernel of step k + 1 (that one has seen every rank announce
 *   step k + 1, i.e. finish reading step k)
 *   svjg_xchg_create   allocates the region of this rank, returns its 64-byte IPC handle
 *   svjg_xchg_open     maps a peer's region from its handle (exchange the handles out of band,
 *                      e.g. torch.distributed.all_gather_object); _close unmaps it
 *   svjg_xchg_counts   counter buffer `parity` (taken modulo 3) of a region: pass it to svjg_filter_reset /
 *                      svjg_filter_device as d_counts
 *   svjg_xchg_signal   after the filter of step `epoch` (1, 2, ...): tells every rank, in stream
 *                      order, that this rank's counters are complete
 *   svjg_genotype_xchg svjg_genotype_device over the sum of all ranks' counters of buffer
 *                      `parity`; waits (on the device) for the signals of step `epoch`;
 *                      signal != 0: the kernel sends this rank's signal itself first (it runs
 *                      behind the filter on the stream), so svjg_xchg_signal is not needed
 *   svjg_xchg_timed_out  1 if a wait gave up after ~2 s (a rank died): results are invalid
 * d_regions[q] is the region of rank q as mapped in THIS process (own region at [rank]). */
int svjg_xchg_create(uint32_t num_sv, void **d_base, uint8_t *ipc_handle64);
int svjg_xchg_open(const uint8_t *ipc_handle64, void **d_peer);
int svjg_xchg_close(void *d_peer);
int svjg_xchg_free(void *d_base);
uint32_t *svjg_xchg_counts(void *d_base, uint32_t num_sv, uint32_t parity);
int svjg_xchg_signal(void *const *d_regions, uint32_t world, uint32_t rank, uint32_t epoch, void *stream);
int svjg_genotype_xchg(void *const *d_regions, uint32_t world, uint32_t rank, uint32_t num_sv, uint32_t parity,
                       uint32_t epoch, int signal, const uint32_t *d_sv_index, const uint8_t *d_svtype, uint32_t n,
                       int64_t min_support, double log10_1me, double log10_e, double log10_half,
                       const double *d_lut, uint32_t lut_nmax, const double *d_k_override, int64_t *d_pl,
                       uint8_t *d_gt, uint32_t *d_ad2, uint8_t *d_flags, void *stream);
int svjg_xchg_timed_out(void *d_base, uint32_t *out);

/* ---- informative_aln.json reader (host) -------------------------------------
 * Replaces predict-genotype.py:67-68 (json.load of <prefix>_informative_aln.json) and
 * :219-226 (nbAln = the lengths of the two lists of a key): the stand-alone
 * predict-genotype front-end gets its counters from the JSON file, as the reference
 * does.  Keys are byte-sorted; counts are [num][2] u32 (UINT32_MAX in both where the
 * value is not "[iterable, iterable, ...]" and the reference would raise on lookup). */
typedef struct svjg_aln_counts svjg_aln_counts;
int svjg_aln_counts_load(const char *json_path, svjg_aln_counts **out);
int svjg_aln_counts_from_memory(const char *json, size_t len, svjg_aln_counts **out);
void svjg_aln_counts_free(svjg_aln_counts *c);
uint32_t svjg_aln_counts_num(const svjg_aln_counts *c);
const char *svjg_aln_counts_key(const svjg_aln_counts *c, uint32_t i, uint32_t *len);
const uint32_t *svjg_aln_counts_data(const svjg_aln_counts *c);
uint32_t svjg_aln_counts_find(const svjg_aln_counts *c, const char *key, uint32_t len);

/* ---- VCF keys and VCF text (host) ---------------------------------------------
 * Replaces the per-record string work of decision_vcf (predict-genotype.py:100-271) around the
 * genotype kernel: svjg_vcf_parse builds, for every body line, the key the reference looks up
 * (:118-211: "chr:DEL-pos-END", "chr:INS-pos-k" with k counted per POS string over all chromosomes,
 * "chr:INV-pos-END", "chr:BND-" + ALT with the REF base replaced by POS, "wrong_format") and the
 * svtype code svjg_genotype_* expects (bit 7 = |length| < 50, :216), keeps the header lines in place
 * (##FORMAT lines dropped, the four FORMAT lines and the column header written for the "#C" line,
 * :102-115) and the first eight columns of the line (:250-256).  `translate_cr` != 0 reads the
 * bytes as text mode does ("\r\n" and a lone "\r" end a line and become "\n"), 0 takes "\n" only
 * (lines already split by the caller).  SVJG_E_INPUT where the reference raises (fewer than 8
 * columns, a missing END=, a non-integer POS/END, a one-piece BND ALT); SVJG_E_UNSUPPORTED for a file
 * with non-ASCII bytes or a POS/END of more than 18 digits (Python's len() / int() semantics are not
 * reproduced for those: use the caller's own string handling).
 * svjg_vcf_index_tables: sv_index[i] for counters that come from the filter (key -> rank among the
 * tables' sv ids).  svjg_vcf_index_counts: the same against an informative_aln.json, plus the
 * svtype array with bit 6 set where the key is present (:216); SVJG_E_INPUT if a gated key's entry is
 * not a pair of lists (:219-226 raises).
 * svjg_vcf_format: the output file's bytes (:248-271) from the kernel's gt / flags / ad2 / pl arrays,
 * in a buffer to release with svjg_buffer_free; *n_genotyped = the "Genotyped svs" count (:275). */
typedef struct svjg_vcf svjg_vcf;
int svjg_vcf_parse(const char *text, size_t len, int translate_cr, svjg_vcf **out);
void svjg_vcf_free(svjg_vcf *v);
uint32_t svjg_vcf_num_records(const svjg_vcf *v);
const uint8_t *svjg_vcf_svtype(const svjg_vcf *v);
const char *svjg_vcf_key(const svjg_vcf *v, uint32_t i, uint32_t *len);   /* NULL: the record has no key */
int svjg_vcf_index_tables(const svjg_vcf *v, const svjg_tables *t, uint32_t *sv_index);
int svjg_vcf_index_counts(const svjg_vcf *v, const svjg_aln_counts *c, uint32_t *sv_index, uint8_t *svtype);
int svjg_vcf_format(const svjg_vcf *v, const uint8_t *gt, const uint8_t *flags, const uint32_t *ad2,
                    const int64_t *pl, char **out, uint64_t *out_len, uint64_t *n_genotyped);
/* svjg_vcf_format_cohort: the text of records [lo, hi) of a multi-sample VCF (svjg_cohort_genotype's arrays of those
 * records, [hi - lo][n_samples]); the pieces of consecutive ranges joined are the whole file.  Every line is the
 * single-sample line with one column per sample, and the column header names the samples: `names` is the names
 * joined by '\t' (names_len bytes).  A range holds the header lines in front of its records and, when hi is the
 * number of records, the ones behind the last.  n_genotyped[s] is ADDED to.  svjg_vcf_format is this with one
 * sample named "SAMPLE". */
int svjg_vcf_format_cohort(const svjg_vcf *v, uint32_t lo, uint32_t hi, uint32_t n_samples, const char *names,
                           uint64_t names_len, const uint8_t *gt, const uint8_t *flags, const uint32_t *ad2,
                           const int64_t *pl, char **out, uint64_t *out_len, uint64_t *n_genotyped);
/* svjg_vcf_format_cohort_tags: svjg_vcf_format_cohort with population INFO tags; svjg_vcf_format_cohort is this with
 * tags = 0 (then gcount, hwe and exchet may be NULL).  `tags` is a mask of SVJG_TAG_*; the tags are written in the
 * order of the bits whatever the mask, with the ##INFO descriptions of bcftools +fill-tags.  gcount [hi - lo][4],
 * hwe and exchet [hi - lo] are svjg_cohort_site_stats's arrays for the range (r0 + h + r2 + m must be n_samples).
 *   NS = r0 + h + r2, AN = 2 NS, AC = h + 2 r2, AF = AC / AN ("." when AN = 0), AC_Het = h, AC_Hom = 2 r2,
 *   F_MISSING = m / S, HWE and ExcHet ("." when NS = 0).  Floats are C's "%.6g" of the double.  The genotype codes
 *   are biallelic: a record whose ALT holds a comma gets "." for the Number=A tags (AC, AF, AC_Het, AC_Hom, HWE,
 *   ExcHet).
 * INFO: the items of the record's INFO (split on ';'; "." or empty is no item) whose key (the text before the first
 * '=') is a selected tag are dropped, the others kept in order, then TAG=value is appended per selected tag.  Header:
 * the catalogue's ##INFO lines of a selected ID are dropped; the new ones are written in front of the ##FORMAT
 * lines.  The bytes do not depend on how the records are cut into ranges. */
#define SVJG_TAG_NS 0x001u
#define SVJG_TAG_AN 0x002u
#define SVJG_TAG_AC 0x004u
#define SVJG_TAG_AF 0x008u
#define SVJG_TAG_AC_HET 0x010u
#define SVJG_TAG_AC_HOM 0x020u
#define SVJG_TAG_F_MISSING 0x040u
#define SVJG_TAG_HWE 0x080u
#define SVJG_TAG_EXCHET 0x100u
int svjg_vcf_format_cohort_tags(const svjg_vcf *v, uint32_t lo, uint32_t hi, uint32_t n_samples, const char *names,
                                uint64_t names_len, const uint8_t *gt, const uint8_t *flags, const uint32_t *ad2,
                                const int64_t *pl, uint32_t tags, const uint32_t *gcount, const double *hwe,
                                const double *exchet, char **out, uint64_t *out_len, uint64_t *n_genotyped);
void svjg_buffer_free(char *p);

/* ---- output (host) ------------------------------------------------------------
 * Replaces filter-alignments.py:174-175: writes json.dumps(dict, sort_keys=True,
 * indent=4) of {sv id: [[ref lines], [alt lines]]} byte-for-byte, from the hit
 * list (any order) and the GAF bytes the offsets refer to. */
int svjg_emit_informative_json(const svjg_tables *t, const uint8_t *gaf, uint64_t n_bytes,
                               const uint32_t *hit_sv2, const uint64_t *hit_off, const uint32_t *hit_len,
                               uint64_t n_hits, const char *out_path);
/* the same text in memory (*out: malloc'd, released with svjg_buffer_free) */
int svjg_emit_informative_json_mem(const svjg_tables *t, const uint8_t *gaf, uint64_t n_bytes, const uint32_t *hit_sv2,
                                   const uint64_t *hit_off, const uint32_t *hit_len, uint64_t n_hits, char **out,
                                   uint64_t *out_len);

#ifdef __cplusplus
}
#endif
#endif /* SVJG_H */
