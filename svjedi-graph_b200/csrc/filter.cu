// Kernels 1-3 of the hot path: GAF ingest (newline scan + field split), alignment
// -> allele resolution through the device link hash, and the per-SV counter /
// hit-tuple reduction.
//
// Reference semantics restated (filter-alignments.py): per-line loop :123-166,
// read_gaf_line :184-198, extract_nodes :351-373, get_aln_links :200-219,
// reverse_link :221-225, check_bkpt_overlap :258-273, get_node_len :343-349.
//
// The work is a chain of three kernels:
//   probe       one block: line length at the head of the shard -> bytes per tile, so that a tile
//               holds about one line per lane of the warp that parses it; zeroes the list cursors.
//   scan        every WARP is an independent worker with its own shared-memory window
//               (no block barrier).  It takes tiles of the byte buffer from a queue (one atomic
//               cursor: a warp that drew node-dense tiles takes fewer); a tile plus 1 KiB of
//               look-ahead is staged by one TMA bulk copy (the warp's next tile is prefetched into L2).
//               A  byte-parallel: every lane classifies 32 bytes with SWAR compares into four
//                  classes (newline, tab, '<'/'>', non-digit); the newlines go straight into the
//                  ordered list of line ends, the others into three bitmaps (tabs, non-digits, node
//                  starts = a byte that is no delimiter right behind one);
//               B  line-parallel: one lane per line reads the line's shape off runs of the tab and
//                  non-digit bitmaps (12 columns, integer columns of digits only, none empty),
//                  counts the path nodes and parses Tlen/Ts/Te of the lines with >= 2 of them;
//               C  node-parallel: one lane per path node of those lines, still from shared
//                  memory: the name is read from its end (digits, '-' or '.', digits, ':', chrom)
//                  with SWAR decimal parses -> exact 24-byte key -> one probe of the plain-node
//                  table (node id, alt length, the roles the node has in link keys);
//               D  same lanes: node-length prefix sums, the breakpoint-overlap verdict of
//                  every link (:269-273), the first-occurrence hazard (:206), and for every link
//                  that can have hits ONE probe of the link table, made by all lanes together;
//                  hit tuples are appended with one cursor atomic per round, counters by RED.
//                  Lines with 33-256 nodes: long_line(), 32 nodes a step.
//               Lines that are not of the plain shape, or do not fit the window, go to the
//               "exact" list.
//   exact       irregular lines.  parse_fields() / general() follow the reference's string
//               semantics literally (odd integers, odd node names, names that could be
//               substrings of earlier ones ...); a regular line that was merely too long for the
//               window gets the fast rules applied where it lies (giant_line()).
// The GAF bytes are read from DRAM once (scan); only the exact route reads them again.
// A line belongs to the tile its first byte is in.
// scan and exact are launched with programmatic stream serialization (launch_pdl): each is scheduled while
// the kernel in front of it finishes, sets up what needs no data of it, then waits for it.
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <map>
#include <mutex>

#include "svjg_internal.h"

namespace cg = cooperative_groups;
using namespace svjg;

namespace {

constexpr int TILE_MIN = 1024;                 // the launch picks the tile so that a tile holds about TILE_LINES lines
constexpr int TILE_LINES = 30;                 // = one line per lane (probe_kernel), within Geo::tile_max
constexpr int LOOKAHEAD = 1024;                // staged behind the tile so that lines starting in it are whole
constexpr int HEAD = 32;                       // staged in front of it (the newline that starts the first line)
constexpr int WARPS = 4;                       // per block; warps never synchronise with each other
constexpr int THREADS = WARPS * 32;
constexpr int SPARE = 32;                      // readable (zero) bytes behind the window

// shared memory of ONE warp of the scan kernel: the window, the newline list, three bitmaps over the
// window's bytes, the lanes of a round's lines.  Two geometries are compiled: MB blocks of WARPS warps per
// SM trade window size (lines per tile, i.e. busy lanes in the line-parallel phase) for resident warps.
template <int MB_, int TILE_MAX_>
struct Geo {
    static constexpr int MB = MB_;                               // blocks per SM the kernel is bounded for
    static constexpr int TILE_MAX = TILE_MAX_;                   // most bytes a warp owns per step, a multiple of 32
    static constexpr int WIN = HEAD + TILE_MAX + LOOKAHEAD;      // window bytes (a multiple of 32, < 64 Ki: offsets are 16 bit)
    static constexpr int NLCAP = WIN / 20 + 1;                   // newline list entries (more newlines in a window => some line is shorter than 20 bytes)
    static constexpr int BMWORDS = WIN / 32 + 3;                 // words per bitmap: reads may run a few words past the window
    static constexpr int OFF_NL = WIN + SPARE;                   // u16[NLCAP]  newline positions, ascending
    static constexpr int OFF_TAB = (OFF_NL + 2 * NLCAP + 15) & ~15;   // u32[BMWORDS]  bit i: window byte i is a tab
    static constexpr int OFF_XD = OFF_TAB + 4 * BMWORDS;         // ... is not '0'..'9'
    static constexpr int OFF_NS = OFF_XD + 4 * BMWORDS;          // ... starts a path node (no '<' / '>', right behind one)
    static constexpr int OFF_TKO = OFF_NS + 4 * BMWORDS;         // u8[32]  lanes of the lines of a round, in order
    static constexpr int OFF_LREC = (OFF_TKO + 32 + 15) & ~15;   // uint2[32]  the multi-node lines of a phase B pass, by lane
    static constexpr int WARP_SMEM = (OFF_LREC + 32 * 8 + 127) & ~127;
    static constexpr int SMEM = WARP_SMEM * WARPS;
    static_assert(TILE_MAX % 32 == 0 && WIN + SPARE < 65536, "window offsets are 16 bit");
    static_assert((SMEM + 1024 + 64) * MB <= 233472, "MB blocks must fit an SM's 228 KB of shared memory");
};
typedef Geo<6, 4992> Geo6;      // 24 warps per SM, tiles of up to ~29 lines of 170 bytes
typedef Geo<8, 3360> Geo8;      // 32 warps per SM, ~21 such lines

constexpr int FLAT_THREADS = 256;              // block size of the flat (grid-stride) kernels

constexpr uint32_t FLAG_EXACT_CHECKS = SVJG_FLAG_EXACT_CHECKS;   // probe links whose overlap test fails too
constexpr uint32_t FLAG_FORCE_GENERAL = SVJG_FLAG_FORCE_GENERAL; // test hook: every multi-node line through general()
constexpr uint32_t FLAG_STOP_AFTER_SCAN = 1u << 8;               // measurement aid: phase A only (SVJG_TUNE_SCAN_ONLY)
constexpr uint32_t COMMA_PATH = 0xFFFFFFFFu;

// device scratch of one svjg_filter_device() call
struct Scratch {
    uint32_t *cnt;        // [2] exact-route lines, [4] bytes per tile, [5] pool cursor, [6] tile queue
    uint32_t *exact;      // line start offsets
    uint4 *slab;          // per warp of the scan kernel: nodes of a long line (long_line())
    uint4 *pool;          // exact kernel: bitmaps and nodes of giant lines, bump-allocated (cnt[5])
    uint32_t cap_exact, cap_pool;
};

struct FilterArgs {
    const uint8_t *gaf;
    uint64_t n;
    uint64_t base;
    int64_t d_over;
    DevTables tb;
    uint32_t *counts;
    uint32_t *hit_sv2, *hit_off, *hit_len;
    uint64_t *hit_off64;         // if set: absolute offsets (base + offset) go here instead of hit_off
    uint64_t hit_cap;
    unsigned long long *stats;   // svjg_filter_stats as 8 x u64
    uint32_t flags;
    uint32_t one;                // 1 (see IsNewline)
    Scratch sc;
    uint32_t skip;               // bytes at the head of the shard that belong to the line in front of it (svjg_filter_json_host)
    uint32_t tile_max;           // most bytes per tile (the scan kernel's geometry)
    uint32_t tile_lines;         // lines a tile should hold (probe_kernel): about one per lane
};

struct Local {
    uint32_t n_rec = 0, n_multi = 0, n_generic = 0;
    uint64_t n_checks = 0;
};

struct GmemSrc {
    typedef uint64_t pos_t;
    const uint8_t *p;
    __device__ __forceinline__ uint32_t operator[](uint64_t i) const { return __ldg(p + i); }
};

__device__ __forceinline__ bool py_space(uint32_t c) {
    return c == ' ' || (c >= 9 && c <= 13) || (c >= 0x1c && c <= 0x1f);
}
__device__ __forceinline__ bool is_delim(uint32_t c) { return (c | 2u) == '>'; }   // '<' = 0x3C, '>' = 0x3E

// aligned 4-byte word of the shard at byte offset al (al % 4 == 0); bytes past the end read as zero
__device__ __forceinline__ uint32_t gaf_word(const FilterArgs &a, uint64_t al) {
    if (al + 4 <= a.n) return __ldg(reinterpret_cast<const uint32_t *>(a.gaf + al));
    uint32_t w = 0;
    for (uint32_t k = 0; k < 4 && al + k < a.n; ++k) w |= uint32_t(__ldg(a.gaf + al + k)) << (8 * k);
    return w;
}

// ---- SWAR byte classes: the answer is bit 7 of each byte, exact for all 256 byte values.
// (w & 0x7F..) ^ C is zero in its low 7 bits iff the byte's low 7 bits equal C; adding 0x7F carries
// into bit 7 unless they are zero; a byte with bit 7 set never matches (C < 0x80).  3 instructions.
#define SVJG_M7 0x7F7F7F7Fu
#define SVJG_H8 0x80808080u
__device__ __forceinline__ uint32_t lop_and_xor(uint32_t w, uint32_t m, uint32_t c) {      // (w & m) ^ c
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0x6A;" : "=r"(r) : "r"(w), "r"(m), "r"(c));
    return r;
}
__device__ __forceinline__ uint32_t lop_nor_and(uint32_t t, uint32_t w, uint32_t h) {      // ~t & ~w & h
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0x02;" : "=r"(r) : "r"(t), "r"(w), "r"(h));
    return r;
}
__device__ __forceinline__ uint32_t lop_or_and(uint32_t t, uint32_t w, uint32_t h) {       // (t | w) & h
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0xA8;" : "=r"(r) : "r"(t), "r"(w), "r"(h));
    return r;
}
__device__ __forceinline__ uint32_t eq_bytes(uint32_t w, uint32_t c4) {                    // c4: four copies of a byte < 0x80
    return lop_nor_and(lop_and_xor(w, SVJG_M7, c4) + SVJG_M7, w, SVJG_H8);
}
// 16 class flags of a 16-byte chunk, bit i = byte i.  dp4a gathers the four bit-7 flags of a
// word: sum(0x80 * weight) = bits << 7.
template <class F>
__device__ __forceinline__ uint32_t mask16(const uint4 &v, F cls) {
    uint32_t lo = __dp4a(cls(v.x), 0x08040201u, 0u);
    lo = __dp4a(cls(v.y), 0x80402010u, lo);
    uint32_t hi = __dp4a(cls(v.z), 0x08040201u, 0u);
    hi = __dp4a(cls(v.w), 0x80402010u, hi);
    return (lo >> 7) | (hi << 1);
}
// 32 class flags of two adjacent 16-byte chunks: four dp4a chains of two words each (8 flags << 7),
// joined by multiply-adds (the fields do not overlap, so + is |)
template <class F>
__device__ __forceinline__ uint32_t mask32(const uint4 &v0, const uint4 &v1, F cls) {
    const uint32_t a0 = __dp4a(cls(v0.y), 0x80402010u, __dp4a(cls(v0.x), 0x08040201u, 0u));
    const uint32_t a1 = __dp4a(cls(v0.w), 0x80402010u, __dp4a(cls(v0.z), 0x08040201u, 0u));
    const uint32_t a2 = __dp4a(cls(v1.y), 0x80402010u, __dp4a(cls(v1.x), 0x08040201u, 0u));
    const uint32_t a3 = __dp4a(cls(v1.w), 0x80402010u, __dp4a(cls(v1.z), 0x08040201u, 0u));
    return (a0 >> 7) + a1 * 2u + a2 * 512u + a3 * 131072u;
}
// The same classes for the byte-parallel phase.  `one` is 1 at run time but opaque to the compiler: the
// carry add becomes an IMAD on the FMA pipe, next to the LOP3s on the ALU pipe (each pipe takes one
// warp instruction every other cycle, so the mix issues faster than ALU work alone).
struct IsNewline {
    uint32_t one;
    __device__ __forceinline__ uint32_t operator()(uint32_t w) const {
        return lop_nor_and(lop_and_xor(w, SVJG_M7, 0x0A0A0A0Au) * one + SVJG_M7, w, SVJG_H8);
    }
};
struct IsTab {
    uint32_t one;
    __device__ __forceinline__ uint32_t operator()(uint32_t w) const {
        return lop_nor_and(lop_and_xor(w, SVJG_M7, 0x09090909u) * one + SVJG_M7, w, SVJG_H8);
    }
};
struct IsNonDigit {
    uint32_t one;
    __device__ __forceinline__ uint32_t operator()(uint32_t w) const {
        return lop_or_and(lop_and_xor(w, SVJG_M7, 0x30303030u) * one + 0x76767676u, w, SVJG_H8);
    }
};
struct IsDelim {
    uint32_t one;
    __device__ __forceinline__ uint32_t operator()(uint32_t w) const {
        return lop_nor_and(lop_and_xor(w, 0x7D7D7D7Du, 0x3C3C3C3Cu) * one + SVJG_M7, w, SVJG_H8);
    }
};

__device__ __noinline__ void report(const FilterArgs &a, uint32_t code, uint64_t line_off) {
    atomicCAS(a.stats + 4, 0ull, (unsigned long long)code);
    atomicMin(a.stats + 5, (unsigned long long)(a.base + line_off));
}

__device__ __forceinline__ void add_stats(const FilterArgs &a, const Local &loc) {
    uint64_t v1 = loc.n_rec, v2 = loc.n_multi, v3 = loc.n_checks, v6 = loc.n_generic;
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        v1 += __shfl_xor_sync(0xFFFFFFFFu, v1, d);
        v2 += __shfl_xor_sync(0xFFFFFFFFu, v2, d);
        v3 += __shfl_xor_sync(0xFFFFFFFFu, v3, d);
        v6 += __shfl_xor_sync(0xFFFFFFFFu, v6, d);
    }
    if ((threadIdx.x & 31) == 0) {
        if (v1) atomicAdd(a.stats + 1, (unsigned long long)v1);
        if (v2) atomicAdd(a.stats + 2, (unsigned long long)v2);
        if (v3) atomicAdd(a.stats + 3, (unsigned long long)v3);
        if (v6) atomicAdd(a.stats + 6, (unsigned long long)v6);
    }
}

// Python int(): optional surrounding whitespace, optional sign, decimal digits.
// (Underscore separators and non-ASCII digits are not accepted: documented.)
template <class Src>
__device__ __noinline__ int parse_int(const Src &src, typename Src::pos_t b, typename Src::pos_t e, int64_t &out) {
    while (b < e && py_space(src[b])) ++b;
    while (e > b && py_space(src[e - 1])) --e;
    bool neg = false;
    if (b < e) {
        uint32_t c = src[b];
        if (c == '+' || c == '-') {
            neg = (c == '-');
            ++b;
        }
    }
    if (b >= e) return SVJG_BAD_INT;
    int64_t v = 0;
    int nd = 0;
    for (; b < e; ++b) {
        uint32_t c = src[b] - '0';
        if (c > 9) return SVJG_BAD_INT;
        if (v != 0 || c != 0) ++nd;
        if (nd > 18) return SVJG_BAD_RANGE;
        v = v * 10 + int64_t(c);
    }
    out = neg ? -v : v;
    return 0;
}

// ---- a whole warp on one long line (exact kernel, one line per warp) ------------------------------
__device__ __forceinline__ uint32_t low_bits(int n);   // the low n bits (defined with the bitmap helpers below)
struct EqByte {
    uint32_t c4;
    __device__ __forceinline__ uint32_t operator()(uint32_t w) const { return eq_bytes(w, c4); }
};
struct DelimByte {
    __device__ __forceinline__ uint32_t operator()(uint32_t w) const {
        return lop_nor_and(lop_and_xor(w, 0x7D7D7D7Du, 0x3C3C3C3Cu) + SVJG_M7, w, SVJG_H8);
    }
};
// class bits of the 16 shard bytes at p (p % 16 == 0); bytes past the end of the shard count as zero
template <class F>
__device__ __forceinline__ uint32_t shard_mask16(const FilterArgs &a, uint64_t p, F cls) {
    uint4 v = make_uint4(0, 0, 0, 0);
    if (p + 16 <= a.n) {
        v = __ldg(reinterpret_cast<const uint4 *>(a.gaf + p));
    } else {
        uint32_t w[4] = {0, 0, 0, 0};
        for (uint32_t k = 0; k < 16 && p + k < a.n; ++k) w[k >> 2] |= uint32_t(__ldg(a.gaf + p + k)) << (8 * (k & 3));
        v = make_uint4(w[0], w[1], w[2], w[3]);
    }
    return mask16(v, cls);
}
// first byte of class `cls` in shard bytes [from, to), all lanes of the warp together; `to` if there is none
template <class F>
__device__ uint64_t coop_find(const FilterArgs &a, uint64_t from, uint64_t to, F cls) {
    const int lane = threadIdx.x & 31;
    for (uint64_t base = from & ~15ull; base < to; base += 512) {
        const uint64_t p = base + 16ull * lane;
        uint32_t m = 0;
        if (p < to) {
            m = shard_mask16(a, p, cls);
            if (p < from) m &= 0xFFFFFFFFu << uint32_t(from - p);
            if (p + 16 > to) m &= low_bits(int(to - p));
        }
        const uint32_t bal = __ballot_sync(0xFFFFFFFFu, m != 0);
        if (bal) {
            const int src = __ffs(bal) - 1;
            return base + 16ull * src + uint32_t(__ffs(__shfl_sync(0xFFFFFFFFu, m, src)) - 1);
        }
    }
    return to;
}
// number of path nodes in [ps, pe): non-delimiter bytes right behind a delimiter (extract_nodes :366-367)
__device__ uint32_t coop_count_nodes(const FilterArgs &a, uint64_t ps, uint64_t pe) {
    const int lane = threadIdx.x & 31;
    uint32_t total = 0, carry = 0;
    for (uint64_t base = ps & ~31ull; base < pe; base += 1024) {
        const uint64_t p = base + 32ull * lane;
        uint32_t d = 0;
        if (p < pe) d = shard_mask16(a, p, DelimByte()) | (shard_mask16(a, p + 16, DelimByte()) << 16);
        uint32_t left = __shfl_up_sync(0xFFFFFFFFu, d, 1) >> 31;           // the byte in front of this lane's 32
        if (lane == 0) left = carry;
        uint32_t st = ((d << 1) | left) & ~d;
        if (p < ps) st &= 0xFFFFFFFFu << uint32_t(ps - p);
        if (p + 32 > pe) st &= low_bits(int(pe > p ? pe - p : 0));
        total += __popc(st);
        carry = __shfl_sync(0xFFFFFFFFu, d, 31) >> 31;
    }
    return __reduce_add_sync(0xFFFFFFFFu, total);
}

// ---------------------------------------------------------------------------
// Rec: one GAF line.  parse_fields()/general() are the exact, string-level
// routines; link()/probe()/emit() are shared with the token-parallel route.
// ---------------------------------------------------------------------------
template <class Src>
struct Rec {
    typedef typename Src::pos_t P;
    const FilterArgs &a;
    Src src;
    P ps, pe;          // path column
    bool angle;
    int64_t tlen, ts, te;
    uint32_t line_off, line_len;
    Local &loc;
    int err;
    bool coop = false;   // all 32 lanes run this line together (exact kernel): long scans are shared

    __device__ Rec(const FilterArgs &a_, Src s, uint32_t off, uint32_t len, Local &l)
        : a(a_), src(s), ps(0), pe(0), angle(true), tlen(0), ts(0), te(0), line_off(off), line_len(len), loc(l), err(0) {}

    struct Tok {
        P b;
        uint32_t l;
    };

    // read_gaf_line (:184-198) on line.rstrip() (:126): 12 tab-separated columns,
    // 9 of them int().  Returns the number of path tokens for a '<'/'>' path,
    // COMMA_PATH for any other non-empty path.  Sets err where the reference raises.
    __device__ __noinline__ uint32_t parse_fields(P s, P e) {
        while (e > s && py_space(src[e - 1])) --e;
        P pos = s;
        int col = 0;
        int64_t alen = 1;
        uint32_t ntok = 0;
        for (;;) {
            P f = pos;
            int r = 0;
            if (col == 5) {
                // path column: find its end and count tokens on the way (extract_nodes :366-367)
                bool prev_delim = true;
                if (coop) {
                    f = P(coop_find(a, uint64_t(pos), uint64_t(e), EqByte{0x09090909u}));
                    ntok = coop_count_nodes(a, uint64_t(pos), uint64_t(f));
                } else
                for (; f < e; ++f) {
                    uint32_t c = src[f];
                    if (c == '\t') break;
                    bool d = is_delim(c);
                    ntok += (prev_delim && !d);
                    prev_delim = d;
                }
                ps = pos;
                pe = f;
            } else {
                uint32_t nd = 0;
                bool plain = true;
                int64_t v = 0;
                for (; f < e; ++f) {
                    uint32_t c = src[f];
                    if (c == '\t') break;
                    uint32_t d = c - '0';
                    plain &= (d <= 9);
                    v = v * 10 + int64_t(d);
                    ++nd;
                }
                bool numeric = (col >= 1 && col <= 3) || (col >= 6 && col <= 11);
                if (numeric) {
                    const bool used = col >= 6 && col <= 8;         // Tlen, Ts, Te: the only values that matter
                    if (!plain || nd == 0 || (nd > 18 && used)) {
                        r = parse_int(src, pos, f, v);
                        // Python's int() has no size limit; only the used columns are held to 18 digits
                        if (r == SVJG_BAD_RANGE && !used) r = 0, v = 1;
                    } else if (nd > 18) {
                        v = 1;                                       // digits only: int() accepts; non-zero unless all '0'
                        bool all0 = true;
                        for (P j = pos; j < f; ++j) all0 &= src[j] == '0';
                        if (all0) v = 0;
                    }
                    if (col == 6) tlen = v;
                    else if (col == 7) ts = v;
                    else if (col == 8) te = v;
                    else if (col == 10) alen = v;
                }
            }
            if (r && !err) err = r;
            ++col;
            if (f >= e || col == 12) break;
            pos = f + 1;
        }
        if (col < 12) err = SVJG_BAD_COLUMNS;
        if (err) return 0;
        if (alen == 0) {                                        // Am / Alen (:196) unless "id:f:" in line (:193)
            bool found = false;
            for (P j = s; j + 5 <= e && !found; ++j)
                found = src[j] == 'i' && src[j + 1] == 'd' && src[j + 2] == ':' && src[j + 3] == 'f' && src[j + 4] == ':';
            if (!found) {
                err = SVJG_BAD_ALEN;
                return 0;
            }
        }
        if (ps == pe) {                                         // p[0] on an empty string (:366)
            err = SVJG_BAD_PATH;
            return 0;
        }
        angle = is_delim(src[ps]);
        return angle ? ntok : COMMA_PATH;
    }

    // tokens of the path column: '<'/'>' separated, or (path not starting with
    // one of those) ','-separated pieces minus their last character
    __device__ bool next_tok(P &cur, Tok &t) const {
        if (angle) {
            while (cur < pe && is_delim(src[cur])) ++cur;
            if (cur >= pe) return false;
            t.b = cur;
            while (cur < pe && !is_delim(src[cur])) ++cur;
            t.l = uint32_t(cur - t.b);
            return true;
        }
        while (cur <= pe) {
            P q = cur;
            while (q < pe && src[q] != ',') ++q;
            P pb = cur;
            uint32_t pl = uint32_t(q - cur);
            cur = q + 1;
            if (pl == 0) continue;
            t.b = pb;
            t.l = pl - 1;
            return true;
        }
        return false;
    }

    __device__ bool tok_eq(const Tok &x, const Tok &y) const {
        if (x.l != y.l) return false;
        if (x.b == y.b) return true;
        for (uint32_t i = 0; i < x.l; ++i)
            if (src[x.b + i] != src[y.b + i]) return false;
        return true;
    }

    __device__ uint64_t tok_hash(const Tok &t) const {
        TokHash h = tok_init();
        uint32_t w = 0;
        for (uint32_t i = 0; i < t.l; ++i) {
            w |= src[t.b + i] << (8 * (i & 3));
            if ((i & 3) == 3) {
                tok_step(h, w);
                w = 0;
            }
        }
        if (t.l & 3) tok_step(h, w);
        return tok_value(h, t.l);
    }

    // name bytes against the table's copy (4-byte aligned, zero padded): word-wide and without an
    // early exit, so all loads are in flight together
    __device__ bool names_match(uint32_t off, const Tok &t) const {
        const uint32_t *q = reinterpret_cast<const uint32_t *>(a.tb.blob + off);
        const uint32_t nw = (t.l + 3u) >> 2;
        const uint64_t al = uint64_t(t.b) & ~3ull;
        const uint32_t sh = (uint32_t(t.b) & 3u) * 8u;
        uint32_t cur = gaf_word(a, al), diff = 0;
#pragma unroll 4
        for (uint32_t k = 0; k < nw; ++k) {
            const uint32_t nxt = gaf_word(a, al + 4ull * (k + 1));
            uint32_t w = __funnelshift_r(cur, nxt, sh);
            cur = nxt;
            if (k == nw - 1 && (t.l & 3u)) w &= (1u << (8u * (t.l & 3u))) - 1u;
            diff |= w ^ __ldg(q + k);
        }
        return diff == 0;
    }

    // node table: name -> (id, alt sequence length); false when the name is in no link key and is
    // no alt node of the GFA
    __device__ bool node_find(uint64_t tokh, const Tok &t, uint32_t &id, int64_t &seq_len) const {
        const uint64_t h = node_hash(tokh);
        uint32_t i = uint32_t(h) & a.tb.node_mask;
        for (;;) {
            const uint4 *sp = reinterpret_cast<const uint4 *>(a.tb.nodes + i);
            const uint4 lo = __ldg(sp), hi = __ldg(sp + 1);
            if (!hi.z) return false;
            const uint64_t sh = (uint64_t(lo.y) << 32) | lo.x;
            if (sh == h && lo.w == t.l && names_match(lo.z, t)) {
                id = hi.z - 1u;
                seq_len = int64_t((uint64_t(hi.y) << 32) | hi.x);
                return true;
            }
            i = (i + 1) & a.tb.node_mask;
        }
    }
    __device__ uint32_t node_id(uint64_t tokh, const Tok &t) const {
        uint32_t id;
        int64_t sl;
        return node_find(tokh, t, id, sl) ? id : NO_NODE;
    }
    // alt_node_len[name] (:346); false when the GFA has no such alt node
    __device__ bool alt_lookup(uint64_t tokh, const Tok &t, int64_t &len) const {
        uint32_t id;
        return node_find(tokh, t, id, len) && len >= 0;
    }

    // link table: exact integer key -> entries
    __device__ bool probe_key(uint64_t key, LinkSlot &out) const {
        uint32_t i = uint32_t(link_hash(key)) & a.tb.link_mask;
        for (;;) {
            const uint4 v = __ldg(reinterpret_cast<const uint4 *>(a.tb.links + i));
            if (!(v.w & 1u)) return false;
            if (((uint64_t(v.y) << 32) | v.x) == key) {
                out.key = key;
                out.val = v.z;
                out.meta = v.w;
                return true;
            }
            i = (i + 1) & a.tb.link_mask;
        }
    }

    // link_kernel stages its hits in shared memory and writes them out with one cursor atomic per
    // block and round; everything else appends to the global arrays directly.
    uint32_t *stage_sv = nullptr, *stage_off = nullptr, *stage_len = nullptr, *stage_n = nullptr;
    uint32_t stage_cap = 0;

    __device__ void emit(uint32_t sv2) {
        if (stage_sv) {
            cg::coalesced_group active = cg::coalesced_threads();
            uint32_t base = 0;
            if (active.thread_rank() == 0) base = atomicAdd(stage_n, active.size());
            base = active.shfl(base, 0) + active.thread_rank();
            if (base < stage_cap) {
                stage_sv[base] = sv2;
                stage_off[base] = line_off;
                stage_len[base] = line_len;
                return;
            }
        }
        // warp-aggregated: one counter atomic per distinct SV allele among the
        // lanes that are here together, one cursor atomic for all of them
        cg::coalesced_group now = cg::coalesced_threads();
        cg::coalesced_group same = cg::labeled_partition(now, sv2);
        if (same.thread_rank() == 0) atomicAdd(a.counts + sv2, same.size());
        unsigned long long base = 0;
        if (now.thread_rank() == 0) base = atomicAdd(a.stats + 0, (unsigned long long)now.size());
        base = now.shfl(base, 0) + now.thread_rank();
        if (base < a.hit_cap) {
            a.hit_sv2[base] = sv2;
            if (a.hit_off64) a.hit_off64[base] = a.base + line_off;
            else a.hit_off[base] = line_off;
            a.hit_len[base] = line_len;
        }
    }

    // forward and reverse key of one link (:141-148) and their entries (:150-166).  idA / idB are
    // the node ids (NO_NODE: the name is in no key, so no key can match).
    // ok_known: the overlap verdict is already there; otherwise it is computed
    // once, on the first key that has entries, by the general overlap().
    // dirs: bit 0 = the forward key can exist, bit 1 = the reverse key can (node roles); 3 = not known
    __device__ void link(const Tok &A, uint32_t idA, int sA, const Tok &B, uint32_t idB, int sB, bool ok_known, bool ok,
                         uint32_t dirs = 3u) {
        if (idA == NO_NODE || idB == NO_NODE) return;
        // one probe where only one key can exist -- the lanes of a warp then probe together whichever
        // key each of them needs; the second probe is for links with both keys possible (forward first)
        const uint64_t fwd = link_key(idA, uint32_t(sA), idB, uint32_t(sB)), rev = link_key(idB, uint32_t(!sB), idA, uint32_t(!sA));
        LinkSlot sl[2];
        bool hit[2];
        hit[0] = dirs != 0u && probe_key((dirs & 1u) ? fwd : rev, sl[0]);
        hit[1] = dirs == 3u && probe_key(rev, sl[1]);
#pragma unroll
        for (int dir = 0; dir < 2; ++dir) {
            if (!hit[dir]) continue;
            const LinkSlot &s = sl[dir];
            if (s.meta & 8u) {
                err = SVJG_BAD_ENTRY;
                return;
            }
            uint32_t cnt = s.meta >> 4;
            if (cnt == 0) continue;
            loc.n_checks += cnt;
            if (!ok_known) {
                ok = overlap(A, B);
                if (err) return;
                ok_known = true;
            }
            if (!ok) continue;
            for (uint32_t k = 0; k < cnt; ++k) {
                uint32_t sv2 = cnt == 1 ? s.val : __ldg(a.tb.entries + s.val + k);
                if (sv2 == ENTRY_POISON) {
                    err = SVJG_BAD_ENTRY;
                    return;
                }
                emit(sv2);
            }
        }
    }

    // ---------------------------------------------------- general (exact) routine
    // strand of a token: the byte in front of the FIRST occurrence of its text
    // anywhere in the path (:206).  1 = '+'.
    __device__ int strand(const Tok &t) {
        if (t.l == 0) {
            err = SVJG_BAD_PATH;
            return 0;
        }
        uint32_t c0 = src[t.b];
        P j = ps;
        for (; j < t.b; ++j) {
            if (src[j] != c0) continue;
            uint32_t i = 1;
            while (i < t.l && src[j + i] == src[t.b + i]) ++i;
            if (i == t.l) break;
        }
        if (j == ps) {
            err = SVJG_BAD_PATH;
            return 0;
        }
        return src[j - 1] == '>';
    }

    // get_node_len (:343-349)
    __device__ int64_t node_len(const Tok &t) {
        P end = t.b + t.l, q = end;
        while (q > t.b && src[q - 1] != ':') --q;
        bool dot = false;
        for (P i = q; i < end; ++i) dot |= (src[i] == '.');
        if (dot) {
            int64_t len = 0;
            if (!alt_lookup(tok_hash(t), t, len)) err = SVJG_BAD_ALTNODE;
            return len;
        }
        P d1 = q;
        while (d1 < end && src[d1] != '-') ++d1;
        if (d1 >= end) {
            err = SVJG_BAD_NODENAME;
            return 0;
        }
        P d2 = d1 + 1;
        while (d2 < end && src[d2] != '-') ++d2;
        int64_t s0, e0;
        int r1 = parse_int(src, d1 + 1, d2, e0);
        int r0 = parse_int(src, q, d1, s0);
        if (r0 || r1) {
            err = (r0 == SVJG_BAD_RANGE || r1 == SVJG_BAD_RANGE) ? SVJG_BAD_RANGE : SVJG_BAD_NODENAME;
            return 0;
        }
        return e0 - s0 + 1;
    }

    // check_bkpt_overlap (:258-273): list.index() picks the FIRST equal node
    __device__ bool overlap(const Tok &A, const Tok &B) {
        P cur = ps;
        Tok t;
        int64_t left = 0, right = 0;
        bool found_l = false, found_r = false;
        while (next_tok(cur, t)) {
            bool is_b = !found_r && tok_eq(t, B);
            if (!found_l || found_r || is_b) {
                int64_t len = node_len(t);
                if (err) return false;
                if (!found_l) {
                    left += len;
                    if (tok_eq(t, A)) found_l = true;
                }
                if (is_b) found_r = true;
                if (found_r) right += len;
            }
        }
        return (left - ts >= a.d_over) && (right - (tlen - te - 1) >= a.d_over);
    }

    // extract_nodes / get_aln_links / lookups for any path (:130-166)
    // `part` of `parts`: the links i with i % parts == part (the lanes of a warp share one heavy line;
    // every node is still the right end of some lane's link, so every strand() is evaluated)
    __device__ __noinline__ void general(uint32_t part = 0, uint32_t parts = 1) {
        uint32_t n = 0;
        {
            P cur = ps;
            Tok t;
            while (next_tok(cur, t)) ++n;
        }
        if (n < 2) return;                                       // :133
        if (part == 0) {
            if (!angle) loc.n_multi++;
            loc.n_generic++;
        }
        P cur = ps;
        Tok A, B;
        next_tok(cur, A);
        uint32_t idA = NO_NODE;
        int sA = 0;
        bool have_a = false;
        for (uint32_t i = 1; i < n; ++i) {
            next_tok(cur, B);
            if (i % parts == part) {
                if (!have_a) {
                    idA = node_id(tok_hash(A), A);
                    sA = strand(A);
                    if (err) return;
                }
                const uint32_t idB = node_id(tok_hash(B), B);
                const int sB = strand(B);
                if (err) return;
                link(A, idA, sA, B, idB, sB, false, false);
                if (err) return;
                idA = idB;
                sA = sB;
                have_a = true;
            } else {
                have_a = false;
            }
            A = B;
        }
    }
};

// ---- TMA bulk copy + mbarrier helpers ---------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// The records are read once: their lines are marked first to leave L2, which keeps the node and link tables there
// (they are what is read again and again)
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    uint64_t once;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(once));
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(once)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// hint: bring [src, src + bytes) into L2 (16-byte aligned, a multiple of 16 bytes)
__device__ __forceinline__ void l2_prefetch(const void *src, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}

__device__ __forceinline__ uint32_t lds32(const uint8_t *win, uint32_t a) { return *reinterpret_cast<const uint32_t *>(win + a); }

// any ',' in window bytes [lo, hi), hi > lo
__device__ __forceinline__ bool has_comma(const uint8_t *win, uint32_t lo, uint32_t hi) {
    const uint32_t a0 = lo & ~3u, a1 = (hi - 1u) & ~3u;
    const uint32_t lom = 0xFFFFFFFFu << (8u * (lo & 3u)), him = 0xFFFFFFFFu >> (8u * (3u - ((hi - 1u) & 3u)));
    uint32_t f = eq_bytes(lds32(win, a0), 0x2C2C2C2Cu) & lom;
    if (a0 == a1) return (f & him) != 0;
    for (uint32_t a = a0 + 4; a < a1; a += 4) f |= eq_bytes(lds32(win, a), 0x2C2C2C2Cu);
    return (f | (eq_bytes(lds32(win, a1), 0x2C2C2C2Cu) & him)) != 0;
}

__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t v, int lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t o = __shfl_up_sync(0xFFFFFFFFu, v, d);
        if (lane >= d) v += o;
    }
    return v;
}

__device__ __forceinline__ uint64_t warp_incl_scan64(uint64_t v, int lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint64_t o = __shfl_up_sync(0xFFFFFFFFu, v, d);
        if (lane >= d) v += o;
    }
    return v;
}

// 32 bits of a byte-indexed bitmap starting at bit `pos`
__device__ __forceinline__ uint32_t bm_bits(const uint32_t *bm, uint32_t pos) {
    const uint32_t w = pos >> 5;
    return __funnelshift_r(bm[w], bm[w + 1], pos & 31u);
}
// the low n bits (n may exceed 32 or be <= 0)
__device__ __forceinline__ uint32_t low_bits(int n) { return __funnelshift_lc(0xFFFFFFFFu, 0u, uint32_t(max(n, 0))); }
// first set bit of the bitmap at or behind `pos` and in front of `end`; `end` (or more) if there is none
__device__ __forceinline__ uint32_t next_tab(const uint32_t *bm, uint32_t pos, uint32_t end) {
    for (uint32_t q = pos; q < end; q += 32) {
        const uint32_t m = bm_bits(bm, q) & low_bits(int(end - q));
        if (m) return q + uint32_t(__ffs(m) - 1);
    }
    return end;
}
// 64 bits of a byte-indexed bitmap starting at bit `pos`; the low n bits of 64
__device__ __forceinline__ uint64_t bm64(const uint32_t *bm, uint32_t pos) {
    const uint32_t w = pos >> 5, sh = pos & 31u;
    const uint32_t b0 = bm[w], b1 = bm[w + 1], b2 = bm[w + 2];
    return (uint64_t(__funnelshift_r(b1, b2, sh)) << 32) | __funnelshift_r(b0, b1, sh);
}
__device__ __forceinline__ uint64_t low_bits64(int n) { return (uint64_t(low_bits(n - 32)) << 32) | low_bits(n); }

// four ASCII digits, the first one in the low byte -> their value (a zero byte counts as '0')
__device__ __forceinline__ uint32_t dec4(uint32_t w) {
    uint32_t t = w & 0x0F0F0F0Fu;
    t = t * 10u + (t >> 8);                     // bytes 0 and 2: two-digit values
    t &= 0x00FF00FFu;
    return (t * 100u + (t >> 16)) & 0xFFFFu;
}
// word with its lowest min(n, 4) bytes cleared (n <= 0: unchanged)
__device__ __forceinline__ uint32_t clear_low_bytes(uint32_t w, int n) {
    return w & __funnelshift_lc(0u, 0xFFFFFFFFu, uint32_t(max(n, 0)) * 8u);
}
// plain-node table: exact key -> (node id, alt sequence length)
__device__ __forceinline__ bool pnode_find(const DevTables &tb, uint64_t c0, uint64_t c1, uint32_t ka, uint32_t kb,
                                           uint32_t &id, uint32_t &alt_len, uint32_t &roles) {
    uint32_t i = pnode_hash(c0, c1, ka, kb) & tb.pnode_mask;
    for (;;) {
        const uint4 *sp = reinterpret_cast<const uint4 *>(tb.pnodes + i);
        const uint4 lo = __ldg(sp), hi = __ldg(sp + 1);
        if (!hi.z) return false;
        if (lo.x == uint32_t(c0) && lo.y == uint32_t(c0 >> 32) && lo.z == uint32_t(c1) && lo.w == uint32_t(c1 >> 32) &&
            hi.x == ka && hi.y == kb) {
            id = (hi.z & PN_ID_MASK) - 1u;
            roles = hi.z >> 28;
            alt_len = hi.w;
            return true;
        }
        i = (i + 1) & tb.pnode_mask;
    }
}

// which of the two keys of a link can exist, from the roles of its nodes: the forward key (A, sA, B, sB)
// needs A as a left node with strand sA and B as a right node with strand sB; the reverse key
// (B, !sB, A, !sA) needs B as a left node with !sB and A as a right node with !sA
__device__ __forceinline__ uint32_t link_dirs(uint32_t rolesA, uint32_t sA, uint32_t rolesB, uint32_t sB) {
    const uint32_t fwd = (rolesA >> sA) & (rolesB >> (2u + sB)) & 1u;
    const uint32_t rev = (rolesB >> (sB ^ 1u)) & (rolesA >> (2u + (sA ^ 1u))) & 1u;
    return fwd | (rev << 1);
}

// ---- byte sources of the node parser: a warp's window in shared memory, or the shard where it lies
struct SmemBytes {
    const uint8_t *p;
    __device__ __forceinline__ uint32_t u8(uint32_t i) const { return p[i]; }
    __device__ __forceinline__ uint32_t u32(uint32_t al) const { return *reinterpret_cast<const uint32_t *>(p + al); }
};
struct ShardBytes {
    const FilterArgs *a;
    __device__ __forceinline__ uint32_t u8(uint32_t i) const { return i < a->n ? __ldg(a->gaf + i) : 0u; }
    __device__ __forceinline__ uint32_t u32(uint32_t al) const { return gaf_word(*a, al); }
};

// the n (1..9) decimal digits that end in front of byte `hi` (validated: digits only)
template <class B>
__device__ __forceinline__ uint32_t dec9(const B &src, uint32_t hi, uint32_t n) {
    const uint32_t base = hi - 8u, al = base & ~3u, sh = (base & 3u) * 8u;
    const uint32_t r0 = src.u32(al), r1 = src.u32(al + 4), r2 = src.u32(al + 8);
    const int m = 8 - int(min(n, 8u));           // bytes of the eight that are not ours
    const uint32_t g0 = dec4(clear_low_bytes(__funnelshift_r(r0, r1, sh), m));
    const uint32_t g1 = dec4(clear_low_bytes(__funnelshift_r(r1, r2, sh), m - 4));
    uint32_t v = g0 * 10000u + g1;
    if (n == 9u) v += (src.u8(hi - 9u) - '0') * 100000000u;
    return v;
}

// ---- phase C: the node whose name is the bytes [tpos, tend) -- exact key, table probe, length.
// Read from the end: digits, '-' or '.', digits, ':', chrom (see PNodeSlot).  xdb: the non-digit bitmap.
struct Node {
    uint32_t nid = NO_NODE;   // node id; NO_NODE: the name is in no link key
    uint32_t nlen = 0;        // get_node_len (:343-349)
    uint32_t akey = 0;        // start value and kind: equal ones in a path mean the first-occurrence rules may bite
    uint32_t roles = 0;       // PNodeSlot roles: bit s = left node of some key with strand s, bit 2+s = right node
    bool plain = false;       // a plain name with a length
};
template <class B>
__device__ __forceinline__ Node resolve_node(const B &src, const uint32_t *xdb, const DevTables &tb, uint32_t tpos, uint32_t tend) {
    Node n;
    const uint32_t L = tend - tpos;
    // non-digit flags of the 32 bytes that end at tend: bit 31 = the last byte of the name; whatever
    // lies in front of the name counts as a non-digit
    const uint32_t Y = bm_bits(xdb, tend - 32u) | low_bits(32 - int(L));
    const uint32_t n2 = uint32_t(__clz(int(Y)));                        // digits of the second number
    const uint32_t n1 = uint32_t(__clz(int(Y << ((n2 + 1u) & 31u))));   // ... of the first (garbage if n2 > 9: rejected)
    const int clen = int(L) - int(n1 + n2 + 2u);                        // bytes in front of the colon
    if (n2 - 1u <= 8u && n1 - 1u <= 8u && uint32_t(clen) <= 15u) {
        const uint32_t q2 = tend - n2, sep = q2 - 1u, q1 = sep - n1, col = q1 - 1u;
        const uint32_t cs = src.u8(sep);
        bool ok = (cs == '-' || cs == '.') && src.u8(col) == ':';
        ok = ok && !(n1 > 1u && src.u8(q1) == '0') && !(n2 > 1u && src.u8(q2) == '0');
        // chrom: the bytes in front of the colon as four words, cleared from the colon on; no second colon
        const uint32_t al = tpos & ~3u, sh = (tpos & 3u) * 8u;
        const uint32_t r0 = src.u32(al), r1 = src.u32(al + 4), r2 = src.u32(al + 8), r3 = src.u32(al + 12), r4 = src.u32(al + 16);
        const uint32_t w0 = __funnelshift_r(r0, r1, sh) & low_bits(8 * clen);
        const uint32_t w1 = __funnelshift_r(r1, r2, sh) & low_bits(8 * clen - 32);
        const uint32_t w2 = __funnelshift_r(r2, r3, sh) & low_bits(8 * clen - 64);
        const uint32_t w3 = (__funnelshift_r(r3, r4, sh) & low_bits(8 * clen - 96)) | (uint32_t(clen) << 24);
        auto has_colon = [](uint32_t w) {
            const uint32_t x = w ^ 0x3A3A3A3Au;
            return (x - 0x01010101u) & ~x & SVJG_H8;
        };
        ok = ok && (has_colon(w0) | has_colon(w1) | has_colon(w2) | has_colon(w3 & 0x00FFFFFFu)) == 0u;
        if (ok) {
            const uint32_t v0 = dec9(src, sep, n1), v1 = dec9(src, tend, n2);
            const uint32_t kind = cs == '.' ? PN_ALT : 0u;
            uint32_t id = NO_NODE, alt_len = PN_NO_LEN;
            const bool found = pnode_find(tb, (uint64_t(w1) << 32) | w0, (uint64_t(w3) << 32) | w2, v0, v1 | kind, id, alt_len, n.roles);
            n.akey = v0 | kind;
            if (!kind) {
                if (v1 >= v0) {                                 // get_node_len :343-349
                    n.plain = true;
                    n.nlen = v1 - v0 + 1u;
                    n.nid = found ? id : NO_NODE;
                }
            } else if (found && alt_len != PN_NO_LEN) {         // alt_node_len[name] :346
                n.plain = true;
                n.nlen = alt_len;
                n.nid = id;
            }
        }
    }
    return n;
}

// the idx-th node start of the path [lps, lpe) in the node-start bitmap (the path has more than idx nodes)
__device__ __forceinline__ uint32_t find_node(const uint32_t *nsb, uint32_t lps, uint32_t idx) {
    uint32_t w = lps >> 5, rem = idx;
    uint32_t bits = nsb[w] & ~low_bits(int(lps & 31u));
    for (;;) {
        const uint32_t c = __popc(bits);
        if (rem < c) break;
        rem -= c;
        bits = nsb[++w];
    }
    for (; rem; --rem) bits &= bits - 1;
    return w * 32u + uint32_t(__ffs(bits) - 1);
}
// first node start at or behind `pos` and in front of `end`; `end` if there is none
__device__ __forceinline__ uint32_t next_node(const uint32_t *nsb, uint32_t pos, uint32_t end) { return next_tab(nsb, pos, end); }

// ---- the links of up to 32 adjacent node pairs, one per lane, all lanes of the warp together: the keys the
// node roles allow are looked up in the link table -- the forward key first, then the reverse one
// (:141-148; a second pass, run only when some link can have both) -- and the entries of the keys found
// become hit tuples, appended with one cursor atomic per pass, and counter increments (:150-166).
// `want`: this lane has a link to look up (both ids known, some key possible, verdict `ok` or exact checks).
__device__ __forceinline__ void probe_links(const FilterArgs &a, bool want, uint32_t idl, uint32_t sl, uint32_t idr, uint32_t sr,
                                            uint32_t dirs, bool ok, uint32_t off, uint32_t len, uint32_t lt_mask, uint32_t &n_checks) {
#pragma unroll 1
    for (uint32_t pass = 0; pass < 2; ++pass) {
        const bool act = want && (pass ? dirs == 3u : dirs != 0u);
        if (pass && !__any_sync(0xFFFFFFFFu, act)) break;
        const bool fwd = pass == 0 && (dirs & 1u);
        const uint32_t kl = fwd ? idl : idr, kr = fwd ? idr : idl, ksl = fwd ? sl : sr ^ 1u, ksr = fwd ? sr : sl ^ 1u;
        const uint32_t key_lo = (kr << 1) | ksr, key_hi = (kl << 1) | ksl;              // link_key() in halves
        uint4 sv = make_uint4(0, 0, 0, 0);
        uint32_t i = link_hash((uint64_t(key_hi) << 32) | key_lo);
        bool go = act, match = false;
        // linear probing: nearly always the first slot settles it (the key, or an empty slot)
        while (__any_sync(0xFFFFFFFFu, go)) {
            if (go) {
                i &= a.tb.link_mask;
                sv = __ldg(reinterpret_cast<const uint4 *>(a.tb.links + i));
                match = (sv.w & 1u) && sv.x == key_lo && sv.y == key_hi;
                go = (sv.w & 1u) && !match;
                ++i;
            }
        }
        const bool poisoned = match && (sv.w & 8u);                      // a key whose value is no list: the reference raises
        const uint32_t cnt = (match && !poisoned) ? sv.w >> 4 : 0u;
        n_checks += cnt;
        const uint32_t mine = ok ? cnt : 0u;                             // tuples of this lane
        uint32_t before, total;
        if (__any_sync(0xFFFFFFFFu, mine > 1u)) {
            const uint32_t incl = warp_incl_scan(mine, int(threadIdx.x & 31));
            before = incl - mine;
            total = __shfl_sync(0xFFFFFFFFu, incl, 31);
        } else {
            const uint32_t hb = __ballot_sync(0xFFFFFFFFu, mine != 0u);
            before = __popc(hb & lt_mask);
            total = __popc(hb);
        }
        if (total) {
            unsigned long long base = 0;
            if ((threadIdx.x & 31) == 0) base = atomicAdd(a.stats + 0, (unsigned long long)total);
            base = __shfl_sync(0xFFFFFFFFu, base, 0) + before;
            for (uint32_t k = 0; k < mine; ++k) {
                const uint32_t sv2 = cnt == 1u ? sv.z : __ldg(a.tb.entries + sv.z + k);
                if (sv2 == ENTRY_POISON) {                               // an entry the reference raises on, reached with ok
                    report(a, SVJG_BAD_ENTRY, off);
                    break;
                }
                atomicAdd(a.counts + sv2, 1u);
                if (base + k < a.hit_cap) {
                    // written once, read by another kernel much later: streaming stores (first to leave L2)
                    __stcs(a.hit_sv2 + base + k, sv2);
                    if (a.hit_off64) __stcs(reinterpret_cast<unsigned long long *>(a.hit_off64) + base + k, (unsigned long long)(a.base + off));
                    else __stcs(a.hit_off + base + k, off);
                    __stcs(a.hit_len + base + k, len);
                }
            }
        }
        if (poisoned) report(a, SVJG_BAD_ENTRY, off);
    }
}

// ---- a line with more path nodes than a warp has lanes: 32 nodes a step.  The first sweep resolves
// the nodes into the warp's slab in device memory (L2) and adds up the lengths; then every node is
// compared with all nodes in front of it (a repeated start value: exact route); the second sweep
// looks the links up.  All lanes call it together; false: the line must take the exact route.
// src / nsb / xdb: the line's bytes and bitmaps -- a warp's window (scan kernel) or the shard itself and
// bitmaps in device memory (exact kernel: giant_line()).
constexpr int SLAB_N = 256;                    // nodes of such a line in the scan kernel (more: exact route)

template <class B>
__device__ __noinline__ bool long_line(const FilterArgs &a, const B src, const uint32_t *nsb, const uint32_t *xdb, uint4 *slab,
                                       uint32_t slab_cap, int lane, uint32_t cnt, uint32_t lps, uint32_t lpe, int64_t lts,
                                       int64_t ltail, uint32_t off, uint32_t len) {
    if (cnt > slab_cap) return false;
    const uint32_t lt_mask = (1u << lane) - 1u;
    uint32_t n_checks = 0;
    uint64_t total = 0;
    bool bad = false;
    uint32_t from = lps;                       // the next step's first node starts at or behind this byte
    for (uint32_t c0 = 0; c0 < cnt; c0 += 32) {
        const bool act = c0 + uint32_t(lane) < cnt;
        Node n;
        uint32_t tpos = lpe, plus = 0;
        if (act) tpos = find_node(nsb, from, uint32_t(lane));
        // the name ends in front of the delimiter of the next node, or with the path
        uint32_t nxt = __shfl_down_sync(0xFFFFFFFFu, tpos, 1);
        if (lane == 31 && act && c0 + 32u < cnt) nxt = next_node(nsb, tpos + 1u, lpe);
        if (act) {
            const uint32_t tend = c0 + uint32_t(lane) + 1u < cnt ? nxt - 1u : lpe;
            plus = src.u8(tpos - 1u) == '>';
            n = resolve_node(src, xdb, a.tb, tpos, tend);
            __stcg(slab + c0 + lane, make_uint4(n.nid, n.nlen, n.akey, plus | (n.roles << 1)));
        }
        bad |= __any_sync(0xFFFFFFFFu, act && !n.plain);
        total += __shfl_sync(0xFFFFFFFFu, warp_incl_scan64(n.nlen, lane), 31);
        from = __shfl_sync(0xFFFFFFFFu, nxt, 31);
    }
    __syncwarp();
    if (bad) return false;
    bool clash = false;
    for (uint32_t c0 = 0; c0 < cnt; c0 += 32) {
        const uint32_t t = c0 + uint32_t(lane);
        const uint32_t mine = t < cnt ? __ldcg(&slab[t].z) : 0u;
        const uint32_t upto = min(c0 + 32u, cnt);
        for (uint32_t j = 0; j < upto; ++j) clash |= j < t && t < cnt && __ldcg(&slab[j].z) == mine;
    }
    if (__any_sync(0xFFFFFFFFu, clash)) return false;
    uint64_t before = 0;
    for (uint32_t c0 = 0; c0 < cnt; c0 += 32) {
        const uint32_t t = c0 + uint32_t(lane);
        const bool act = t < cnt;
        const uint4 me = act ? __ldcg(slab + t) : make_uint4(NO_NODE, 0, 0, 0);
        const uint4 lf = act && t ? __ldcg(slab + t - 1) : make_uint4(NO_NODE, 0, 0, 0);
        const uint64_t incl = warp_incl_scan64(me.y, lane);
        const uint64_t pre = before + incl - me.y;
        const bool ok = (int64_t(pre) - lts >= a.d_over) && (int64_t(total - pre) - ltail >= a.d_over);
        const uint32_t dirs = link_dirs(lf.w >> 1, lf.w & 1u, me.w >> 1, me.w & 1u);
        const bool want = act && t && lf.x != NO_NODE && me.x != NO_NODE && dirs && (ok || (a.flags & FLAG_EXACT_CHECKS));
        probe_links(a, want, lf.x, lf.w & 1u, me.x, me.w & 1u, dirs, ok, off, len, lt_mask, n_checks);
        before += __shfl_sync(0xFFFFFFFFu, incl, 31);
    }
    n_checks = __reduce_add_sync(0xFFFFFFFFu, n_checks);
    if (lane == 0 && n_checks) atomicAdd(a.stats + 3, (unsigned long long)n_checks);
    return true;
}

// ===========================================================================
// scan: newline scan, column split, validation, path walk, node and link resolution, hits
// ===========================================================================
template <class G>
__global__ void __launch_bounds__(THREADS, G::MB) scan_kernel(const __grid_constant__ FilterArgs a) {
    extern __shared__ __align__(128) uint8_t smem_all[];
    __shared__ __align__(8) uint64_t mbars[WARPS];
    __shared__ uint32_t next_tile[WARPS];                                  // the tile each warp takes next

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t lt_mask = (1u << lane) - 1u;
    uint8_t *win = smem_all + warp * G::WARP_SMEM;                         // the window; everything else at fixed offsets behind it
    uint16_t *nl = reinterpret_cast<uint16_t *>(win + G::OFF_NL);          // newline positions, ascending
    uint32_t *tabb = reinterpret_cast<uint32_t *>(win + G::OFF_TAB);       // bit i: window byte i is a tab
    uint32_t *xdb = reinterpret_cast<uint32_t *>(win + G::OFF_XD);         // bit i: ... is not '0'..'9'
    uint32_t *nsb = reinterpret_cast<uint32_t *>(win + G::OFF_NS);         // bit i: ... starts a path node
    uint8_t *tko = win + G::OFF_TKO;
    uint2 *lrec = reinterpret_cast<uint2 *>(win + G::OFF_LREC);            // {s | line bytes << 16, ps | pe << 16}
    uint64_t *mbar = &mbars[warp];
    const SmemBytes src{win};

    if (lane == 0) mbar_init(mbar, 1);
    for (int i = lane; i < G::BMWORDS; i += 32) tabb[i] = 0, xdb[i] = 0, nsb[i] = 0;
    for (int i = G::WIN + lane; i < G::WIN + SPARE; i += 32) win[i] = 0;   // never written by the copies
    __syncwarp();
    uint32_t phase = 0;
    uint32_t u_rec = 0, u_multi = 0, n_checks = 0;   // tallies: lines, lines with >= 2 nodes (both warp-uniform), overlap tests
    const uint32_t one = a.one;
    const uint32_t n_workers = gridDim.x * WARPS;

    cudaGridDependencySynchronize();                               // probe_kernel: the tile size, zeroed cursors
    cudaTriggerProgrammaticLaunchCompletion();                     // exact_kernel may be scheduled as blocks retire
    const uint32_t tile_bytes = a.sc.cnt[4];                       // chosen by probe_kernel: a multiple of 32, at most G::TILE_MAX
    const uint32_t n_tiles = uint32_t((a.n + tile_bytes - 1) / tile_bytes);
    const uint32_t win_bytes = HEAD + tile_bytes + LOOKAHEAD, n_pairs = win_bytes / 32u;

    // The first tile of every warp is fixed, the rest come from the queue cnt[6] (tiles n_workers, n_workers + 1, ...):
    // a warp that drew slow tiles takes fewer, and the SMs run out of work together.
    for (uint32_t tile = blockIdx.x * WARPS + warp; tile < n_tiles; tile = next_tile[warp], __syncwarp()) {
        const uint64_t tile_start = uint64_t(tile) * tile_bytes;
        const uint64_t g0 = tile_start ? tile_start - HEAD : 0;
        const uint32_t dst0 = tile_start ? 0 : HEAD;
        uint64_t g1 = tile_start + tile_bytes + LOOKAHEAD;
        if (g1 > a.n) g1 = a.n;
        const bool at_eof = (g1 == a.n);
        const uint32_t nbytes = uint32_t(g1 - g0);
        const uint32_t bulk = nbytes & ~15u;
        const uint32_t valid_end = dst0 + nbytes;
        const uint32_t wbase = uint32_t(tile_start) - HEAD;            // shard offset = wbase + window offset

        if (lane == 0) {
            if (bulk) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                mbar_expect_tx(mbar, bulk);
                bulk_g2s(win + dst0, a.gaf + g0, bulk, mbar);
            }
            // the tile this warp takes next, drawn while the copy is in flight: on its way into L2 while this one is parsed
            const uint32_t next = n_workers + atomicAdd(a.sc.cnt + 6, 1u);
            next_tile[warp] = next;                                // read behind the tile's last __syncwarp()
            const uint64_t nx = uint64_t(next) * tile_bytes;
            if (nx + tile_bytes + LOOKAHEAD <= a.n) l2_prefetch(a.gaf + nx - HEAD, win_bytes);
        }
        if (bulk != nbytes || dst0 || valid_end < win_bytes) {                       // the first and the last tiles of the shard
            for (uint32_t i = bulk + lane; i < nbytes; i += 32) win[dst0 + i] = __ldg(a.gaf + g0 + i);
            if (dst0) win[lane] = (lane == HEAD - 1 && a.skip == 0u) ? '\n' : 0;   // "newline" in front of byte 0 of the file
            for (uint32_t i = valid_end + lane; i < win_bytes; i += 32) win[i] = 0;
        }
        if (bulk) {
            mbar_wait(mbar, phase);
            phase ^= 1;
        }
        __syncwarp();

        // ---- phase A: byte classes.  A lane takes two adjacent 16-byte chunks = one word of each bitmap;
        // the newlines go straight into the ordered list.  The scan stops behind the tile once the last
        // owned line has its end.
        const uint32_t own_end = min(HEAD + tile_bytes, valid_end);   // lines starting before own_end are ours
        uint32_t n_nl = 0, n_own = 0;
        for (uint32_t c0 = 0; c0 < n_pairs; c0 += 32) {
            const uint32_t c = c0 + uint32_t(lane);
            const uint32_t p0 = c * 32u;
            uint32_t m = 0;
            if (c < n_pairs) {
                const uint4 v0 = *reinterpret_cast<const uint4 *>(win + p0);
                const uint4 v1 = *reinterpret_cast<const uint4 *>(win + p0 + 16);
                m = mask32(v0, v1, IsNewline{one});
                tabb[c] = mask32(v0, v1, IsTab{one});
                xdb[c] = mask32(v0, v1, IsNonDigit{one});
                const uint32_t d = mask32(v0, v1, IsDelim{one});
                const uint32_t left = c ? uint32_t(is_delim(win[p0 - 1u])) : 0u;     // the byte in front of these 32
                nsb[c] = ((d << 1) | left) & ~d;
                if (c == 0) m &= 0x80000000u;                             // positions before HEAD-1 are not ours to see
            }
            // newline positions, in order: one per 32 bytes as a rule
            if (__any_sync(0xFFFFFFFFu, (m & (m - 1u)) != 0u)) {
                // two line ends in 32 bytes (hardly ever): the general placement
                const uint32_t cnt = __popc(m), incl = warp_incl_scan(cnt, lane);
                uint32_t idx = n_nl + incl - cnt, own = 0;
                for (uint32_t mm = m; mm; mm &= mm - 1) {
                    const uint32_t pos = p0 + uint32_t(__ffs(mm) - 1);
                    if (idx < uint32_t(G::NLCAP)) nl[idx] = uint16_t(pos);
                    own += pos + 1u < own_end;
                    ++idx;
                }
                n_nl += __shfl_sync(0xFFFFFFFFu, incl, 31);
                n_own += __reduce_add_sync(0xFFFFFFFFu, own);
            } else {
                const uint32_t pos = p0 + uint32_t(__ffs(m)) - 1u;                 // if this lane has one
                const uint32_t b = __ballot_sync(0xFFFFFFFFu, m != 0u);
                const uint32_t bo = __ballot_sync(0xFFFFFFFFu, m != 0u && pos + 1u < own_end);   // ... that starts an owned line
                const uint32_t idx = n_nl + __popc(b & lt_mask);
                if (m != 0u && idx < uint32_t(G::NLCAP)) nl[idx] = uint16_t(pos);
                n_nl += __popc(b);
                n_own += __popc(bo);
            }
            // behind the tile: a newline at or after own_end - 1 ends the last owned line
            if ((c0 + 32u) * 32u >= own_end && __any_sync(0xFFFFFFFFu, (m & ~low_bits(int(own_end) - 1 - int(p0))) != 0)) break;
        }
        __syncwarp();
        if (a.flags & FLAG_STOP_AFTER_SCAN) continue;                 // measurement aid (SVJG_TUNE_SCAN_ONLY)

        if (n_nl > uint32_t(G::NLCAP)) {
            // that many lines in the window: some line is shorter than 20 bytes and cannot hold 12 columns
            if (lane == 0) report(a, SVJG_BAD_SHORTLINE, tile_start);
            __syncwarp();
            continue;
        }
        u_rec += n_own;
        // ---- phase B: one lane per line, mostly bit work on the class bitmaps
        for (uint32_t k0 = 0; k0 < n_own; k0 += 32) {
            const uint32_t k = k0 + lane;
            uint32_t want = 0;                 // path nodes of a plain line with >= 2 of them
            bool exact = false;                // the line must take the exact route
            uint32_t s = 0, e = 0, ps = 0, pe = 0;
            uint32_t c6 = 0, c7 = 0, c8 = 0, c9 = 0;   // tabs that end columns 6-9
            bool has_nl = false;
            if (k < n_own) {
                s = uint32_t(nl[k]) + 1u;
                if (k + 1 < n_nl) {
                    e = nl[k + 1];
                    has_nl = true;
                } else if (at_eof) {
                    e = valid_end;
                } else {
                    exact = true;              // runs past the window
                }
                if (!exact) {
                    // Shape of a plain line, read off the tab bitmap and the non-digit bitmap:
                    //   name TAB digits TAB digits TAB digits TAB strand TAB path TAB (digits TAB) x 5 digits [TAB tags]
                    // A run of digits and single tabs must follow the first tab up to the strand, and the
                    // sixth tab up to the tags (or the end of the line).  Anything else: the exact route.
                    bool plain = e > s && !py_space(win[e - 1]);
                    uint32_t t1;
                    {
                        const uint64_t t64 = bm64(tabb, s) & low_bits64(int(e - s));      // a read name is rarely longer
                        t1 = t64 ? s + uint32_t(__ffsll((long long)t64)) - 1u : next_tab(tabb, min(s + 64u, e), e);
                    }
                    plain &= t1 < e;
                    const uint32_t n2 = t1 + 1u;                                          // first byte of column 2
                    const uint32_t tw = bm_bits(tabb, n2);
                    const uint32_t xa = bm_bits(xdb, n2) & ~tw;                           // neither digit nor tab (the newline is one)
                    plain &= xa != 0;
                    const uint32_t l2 = uint32_t(__ffs(xa)) - 1u;                         // length of the run: columns 2-4 and their tabs
                    const uint32_t ta = tw & low_bits(int(l2));
                    // tabs 2, 3 and 4 and nothing else, the last one right in front of the strand, no empty column
                    plain &= __popc(ta) == 3 && (ta >> ((l2 - 1u) & 31u)) == 1u && (ta & ((ta >> 1) | 1u)) == 0;
                    const uint32_t n5 = n2 + l2;                                          // strand
                    // a one-byte strand column as a rule: its tab is in the bits at hand
                    ps = (l2 < 31u && ((tw >> (l2 + 1u)) & 1u)) ? n5 + 2u : next_tab(tabb, min(n5, e), e) + 1u;
                    // the path column ends at the next tab; its node starts are counted on the way
                    uint32_t ntok = 0;
                    pe = e;
                    for (uint32_t q = ps; q < e; q += 32) {
                        const uint32_t tb = bm_bits(tabb, q) & low_bits(int(e - q));
                        const uint32_t nb = bm_bits(nsb, q);
                        if (tb) {
                            const uint32_t r = uint32_t(__ffs(tb)) - 1u;
                            pe = q + r;
                            ntok += __popc(nb & low_bits(int(r)));
                            break;
                        }
                        ntok += __popc(nb);
                    }
                    plain &= pe < e && pe > ps;
                    const uint32_t n7 = min(pe + 1u, e);                                  // first byte of column 7
                    uint64_t tt = bm64(tabb, n7);
                    const uint64_t xt = bm64(xdb, n7) & ~tt;
                    plain &= xt != 0;
                    const uint32_t l7 = uint32_t(__ffsll((long long)xt)) - 1u;            // length of the run: columns 7-12 and their tabs
                    tt &= low_bits64(int(l7));
                    const uint32_t ntab = uint32_t(__popcll(tt));
                    const bool last_is_tab = l7 != 0 && ((tt >> ((l7 - 1u) & 63u)) & 1ull) != 0;
                    // six tabs, the sixth right in front of the tags -- or five and the line ends behind column 12
                    plain &= (ntab == 6 && last_is_tab) || (ntab == 5 && !last_is_tab && n7 + l7 == e);
                    plain &= (tt & ((tt >> 1) | 1ull)) == 0;                              // no empty column
                    // tabs 7-10: the coordinates are columns 7-9, Alen (column 11, behind tab 10) must not start with '0'
                    c6 = pe;
                    c7 = n7 + uint32_t(__ffsll((long long)tt)) - 1u;
                    tt &= tt - 1;
                    c8 = n7 + uint32_t(__ffsll((long long)tt)) - 1u;
                    tt &= tt - 1;
                    c9 = n7 + uint32_t(__ffsll((long long)tt)) - 1u;
                    tt &= tt - 1;
                    const uint32_t p10 = n7 + uint32_t(__ffsll((long long)tt)) - 1u;
                    plain = plain && win[p10 + 1] != '0';
                    if (!plain) {
                        exact = true;
                    } else if (!is_delim(win[ps])) {
                        // bare name or GFA-style a+,b+ (extract_nodes :369-373): one piece without ',' is one node
                        exact = has_comma(win, ps, pe);
                    } else if (ntok >= 2) {                                                // :133
                        if (a.flags & FLAG_FORCE_GENERAL) exact = true;
                        else want = ntok;
                    }
                }
            }
            __syncwarp();
            // Tlen, Ts, Te of the lines that go on (digit-only columns 7-9): values of up to nine digits here,
            // anything longer (a path of a billion bases) is the exact route's
            int32_t ts = 0, tail = 0;
            if (want) {
                const uint32_t n_tlen = c7 - c6 - 1u, n_ts = c8 - c7 - 1u, n_te = c9 - c8 - 1u;
                if (max(n_tlen, max(n_ts, n_te)) <= 9u) {
                    ts = int32_t(dec9(src, c8, n_ts));
                    tail = int32_t(dec9(src, c7, n_tlen)) - int32_t(dec9(src, c9, n_te)) - 1;
                    lrec[lane] = make_uint2(s | ((e - s + (has_nl ? 1u : 0u)) << 16), ps | (pe << 16));
                } else {
                    exact = true;
                    want = 0;
                }
            }
            __syncwarp();
            // ---- phases C and D: rounds of at most 32 path nodes, whole lines only, one lane per node
            uint32_t pend = want > 32u ? 0u : want;
            while (__any_sync(0xFFFFFFFFu, pend != 0)) {
                const uint32_t incl = warp_incl_scan(pend, lane);
                const bool take = pend != 0 && incl <= 32u;                     // a prefix of the pending lines
                const uint32_t takeb = __ballot_sync(0xFFFFFFFFu, take);
                const uint32_t ntk = __shfl_sync(0xFFFFFFFFu, incl, 31 - __clz(takeb));
                const uint32_t first = incl - pend;                             // list slot of this line's first node
                // no list of nodes is written: a node lane finds its line from the bit mask of the lines'
                // first slots, and its own start in the node-start bitmap
                const uint32_t startmask = __reduce_or_sync(0xFFFFFFFFu, take ? (1u << first) : 0u);
                if (take) tko[__popc(takeb & lt_mask)] = uint8_t(lane);             // ordinal among the taken lines -> lane
                __syncwarp();
                const bool is_tok = uint32_t(lane) < ntk;
                uint32_t own_l = 0, idx = 0;
                if (is_tok) {
                    const uint32_t below = startmask & (0xFFFFFFFFu >> (31 - lane));
                    own_l = tko[__popc(below) - 1];
                    idx = uint32_t(lane) - uint32_t(31 - __clz(below));             // number of this node in its line
                }
                const uint2 lr = lrec[own_l];
                const uint32_t lpath = lr.y;
                const uint32_t lcnt = __shfl_sync(0xFFFFFFFFu, pend, own_l);
                // C: this lane's node; its name ends in front of the next node's delimiter, or with the path
                uint32_t tpos = 0;
                if (is_tok) tpos = find_node(nsb, lpath & 0xFFFFu, idx);
                const uint32_t nxt = __shfl_down_sync(0xFFFFFFFFu, tpos, 1);
                Node nd;
                uint32_t plus = 0;
                if (is_tok) {
                    plus = win[tpos - 1u] == '>';
                    nd = resolve_node(src, xdb, a.tb, tpos, idx + 1u < lcnt ? nxt - 1u : lpath >> 16);
                }
                const uint32_t nid = nd.nid, nlen = nd.nlen, akey = nd.akey;
                // D: per line -- sums of the node lengths left of every node, names that repeat a start
                // value (the first-occurrence rules :206 and :269-271 bite), verdicts
                const uint32_t lfirst = uint32_t(lane) - idx;
                // a repeated start value: some other lane of the line holds the same key (one MATCH)
                const uint32_t line_lanes = low_bits(int(lcnt)) << lfirst;
                const uint32_t twins = __match_any_sync(0xFFFFFFFFu, akey) & line_lanes;
                bool clash = (twins & ~(1u << lane)) != 0;
                // segmented inclusive scan of the lengths: a lane adds what lies `d` to its left while
                // that is still its own line
                uint64_t lsum = nlen;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint64_t o = __shfl_up_sync(0xFFFFFFFFu, lsum, d);
                    if (uint32_t(d) <= idx) lsum += o;
                }
                // left of a link = the nodes up to and with its left node, right = from its right node on (:269-271)
                uint64_t pre_l = lsum - nlen, pre_r = pre_l;
                uint32_t splus = plus, sl = __shfl_up_sync(0xFFFFFFFFu, plus, 1);
                if (__any_sync(0xFFFFFFFFu, is_tok && clash)) {
                    // The same NAME again (a read through both ends of a breakend in one node): the reference takes
                    // the strand of a name from its first occurrence in the path (:206) and sums the lengths up to /
                    // from its first index (nodes.index, :269-271) -- the lane of the first twin has both (a lane
                    // without twins is its own first).  Twins that are different names with one start value (one
                    // may be a substring of the other) stay with the exact route.
                    const int twin0 = is_tok ? __ffs(twins) - 1 : lane;
                    const uint32_t f_nid = __shfl_sync(0xFFFFFFFFu, nid, twin0);
                    const uint64_t f_sum = __shfl_sync(0xFFFFFFFFu, lsum, twin0);
                    const uint32_t f_len = __shfl_sync(0xFFFFFFFFu, nlen, twin0);
                    splus = __shfl_sync(0xFFFFFFFFu, plus, twin0);
                    sl = __shfl_up_sync(0xFFFFFFFFu, splus, 1);
                    pre_l = __shfl_up_sync(0xFFFFFFFFu, f_sum, 1);           // through the first occurrence of the left node
                    pre_r = f_sum - f_len;                                   // in front of the first occurrence of this one
                    clash = clash && !(nid != NO_NODE && f_nid == nid);
                }
                const uint32_t bad = __reduce_or_sync(0xFFFFFFFFu, (is_tok && (!nd.plain || clash)) ? (1u << own_l) : 0u);
                const uint64_t total = __shfl_sync(0xFFFFFFFFu, lsum, is_tok ? lfirst + lcnt - 1u : 0u);
                const uint32_t idl = __shfl_up_sync(0xFFFFFFFFu, nid, 1);
                const int64_t lts = __shfl_sync(0xFFFFFFFFu, ts, own_l), ltail = __shfl_sync(0xFFFFFFFFu, tail, own_l);
                const uint32_t loff = wbase + (lr.x & 0xFFFFu), llen = lr.x >> 16;
                const bool ok = (int64_t(pre_l) - lts >= a.d_over) && (int64_t(total - pre_r) - ltail >= a.d_over);
                const uint32_t dirs = link_dirs(__shfl_up_sync(0xFFFFFFFFu, nd.roles, 1), sl, nd.roles, splus);
                const bool look = is_tok && idx >= 1 && !((bad >> own_l) & 1u) && idl != NO_NODE && nid != NO_NODE && dirs &&
                                  (ok || (a.flags & FLAG_EXACT_CHECKS));
                probe_links(a, look, idl, sl, nid, splus, dirs, ok, loff, llen, lt_mask, n_checks);
                if (take) {
                    if ((bad >> lane) & 1u) exact = true;
                    pend = 0;
                }
                u_multi += __popc(takeb & ~bad);
                __syncwarp();
            }
            // ---- lines with more nodes than a round has lanes: one line at a time (long_line())
            for (uint32_t longb = __ballot_sync(0xFFFFFFFFu, want > 32u); longb; longb &= longb - 1) {
                const int L = __ffs(longb) - 1;
                const uint2 lr = lrec[L];
                const bool done = long_line(a, src, nsb, xdb, a.sc.slab + size_t(blockIdx.x * WARPS + warp) * SLAB_N, SLAB_N, lane,
                                            __shfl_sync(0xFFFFFFFFu, want, L), lr.y & 0xFFFFu, lr.y >> 16,
                                            __shfl_sync(0xFFFFFFFFu, ts, L), __shfl_sync(0xFFFFFFFFu, tail, L),
                                            wbase + (lr.x & 0xFFFFu), lr.x >> 16);
                if (!done && lane == L) exact = true;
                u_multi += done;
            }
            const uint32_t xb = __ballot_sync(0xFFFFFFFFu, exact);
            if (xb) {
                uint32_t xbase = 0;
                if (lane == 0) xbase = atomicAdd(a.sc.cnt + 2, uint32_t(__popc(xb)));
                xbase = __shfl_sync(0xFFFFFFFFu, xbase, 0);
                if (exact) {
                    const uint32_t idx = xbase + __popc(xb & lt_mask);
                    if (idx < a.sc.cap_exact) a.sc.exact[idx] = wbase + s;
                    else report(a, SVJG_BAD_SHORTLINE, wbase + s);   // only possible with lines shorter than 16 bytes
                }
            }
        }
        __syncwarp();
    }
    n_checks = __reduce_add_sync(0xFFFFFFFFu, n_checks);
    if (lane == 0) {
        if (u_rec) atomicAdd(a.stats + 1, (unsigned long long)u_rec);
        if (u_multi) atomicAdd(a.stats + 2, (unsigned long long)u_multi);
        if (n_checks) atomicAdd(a.stats + 3, (unsigned long long)n_checks);
    }
}

// ===========================================================================
// exact: one thread per irregular line — the reference's string semantics, literally
// ===========================================================================
// A line that is regular but too long for the scan kernel's window (thousands of path nodes): the warp
// builds the node-start and non-digit bitmaps of its path column in device memory and runs long_line() on
// the bytes where they lie.  false: general() decides.
__device__ __noinline__ bool giant_line(const FilterArgs &a, uint32_t ps, uint32_t pe, uint32_t ntok, int64_t ts, int64_t tail,
                                        uint32_t off, uint32_t len, int lane, Local &loc) {
    if (ps < 64u) return false;                                             // the node parser looks 32 bytes back
    const uint32_t w0 = (ps >> 5) - 1u, nw = (pe >> 5) - w0 + 4u;          // bitmap words, a few to spare on both sides
    const uint32_t bm16 = (nw + 3u) / 4u;                                   // one bitmap in 16-byte units
    const uint32_t need = 2u * bm16 + ntok;                                 // two bitmaps, then one unit per node
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(a.sc.cnt + 5, need);
    base = __shfl_sync(0xFFFFFFFFu, base, 0);
    if (uint64_t(base) + need > a.sc.cap_pool) return false;
    uint32_t *nsb = reinterpret_cast<uint32_t *>(a.sc.pool + base), *xdb = reinterpret_cast<uint32_t *>(a.sc.pool + base + bm16);
    for (uint32_t w = uint32_t(lane); w < nw; w += 32) {
        const uint64_t pos = uint64_t(w0 + w) * 32u;
        uint32_t d = 0, x = 0;
        if (pos + 32 <= a.n) {
            const uint4 v0 = __ldg(reinterpret_cast<const uint4 *>(a.gaf + pos)), v1 = __ldg(reinterpret_cast<const uint4 *>(a.gaf + pos + 16));
            d = mask16(v0, IsDelim{1u}) | (mask16(v1, IsDelim{1u}) << 16);
            x = mask16(v0, IsNonDigit{1u}) | (mask16(v1, IsNonDigit{1u}) << 16);
        } else {
            for (uint32_t k = 0; k < 32; ++k) {
                const uint32_t c = pos + k < a.n ? uint32_t(__ldg(a.gaf + pos + k)) : 0u;
                d |= uint32_t(is_delim(c)) << k;
                x |= uint32_t(c - '0' > 9u) << k;
            }
        }
        const uint32_t left = uint32_t(is_delim(__ldg(a.gaf + pos - 1)));   // pos >= 32
        __stcg(nsb + w, ((d << 1) | left) & ~d);
        __stcg(xdb + w, x);
    }
    __syncwarp();
    return long_line(a, ShardBytes{&a}, nsb - w0, xdb - w0, a.sc.pool + base + 2u * bm16, ntok, lane, ntok, ps, pe, ts, tail, off, len);
}

__global__ void __launch_bounds__(FLAT_THREADS) exact_kernel(const __grid_constant__ FilterArgs a) {
    cudaGridDependencySynchronize();                               // scan_kernel: the list and its length
    cudaTriggerProgrammaticLaunchCompletion();
    const uint32_t n = min(a.sc.cnt[2], a.sc.cap_exact);
    if (n == 0) return;                                            // the rule on regular input: nothing to set up
    Local loc;
    // Lines differ wildly in the work they need (general() is quadratic in the path nodes), and lanes
    // of a warp that run different lines execute one after the other.  While there are few lines,
    // every line gets a warp of its own and the lanes share its links; only a flood of them goes one
    // line per thread.
    const uint32_t n_warps = gridDim.x * (FLAT_THREADS / 32);
    const bool per_warp = n <= 4u * n_warps;
    const uint32_t me = per_warp ? (blockIdx.x * FLAT_THREADS + threadIdx.x) >> 5 : blockIdx.x * FLAT_THREADS + threadIdx.x;
    const uint32_t stride = per_warp ? n_warps : gridDim.x * FLAT_THREADS;
    const uint32_t part = per_warp ? (threadIdx.x & 31u) : 0u, parts = per_warp ? 32u : 1u;
    if (blockIdx.x == 0 && threadIdx.x == 0 && n) atomicAdd(a.stats + 7, (unsigned long long)n);
    for (uint32_t i = me; i < n; i += stride) {
        const uint32_t off = a.sc.exact[i];
        uint64_t e = off;
        if (per_warp) e = coop_find(a, off, a.n, EqByte{0x0A0A0A0Au});
        else
            while (e < a.n && __ldg(a.gaf + e) != '\n') ++e;
        const uint32_t len = uint32_t(e - off) + (e < a.n ? 1u : 0u);
        Rec<GmemSrc> rec(a, GmemSrc{a.gaf}, off, len, loc);
        rec.coop = per_warp;
        const uint32_t ntok = rec.parse_fields(uint64_t(off), e);
        if (!rec.err && ntok >= 2) {
            if (ntok != COMMA_PATH && part == 0) loc.n_multi++;
            // a warp of its own: first the fast rules on the bytes where they lie; if they do not apply, general()
            const bool fast = per_warp && ntok != COMMA_PATH && !(a.flags & FLAG_FORCE_GENERAL) && e < 0xFFFFFFFFull &&
                              giant_line(a, uint32_t(rec.ps), uint32_t(rec.pe), ntok, rec.ts, rec.tlen - rec.te - 1, off, len,
                                         int(threadIdx.x & 31u), loc);
            if (!fast) rec.general(part, parts);
        }
        if (rec.err) report(a, rec.err, off);
    }
    add_stats(a, loc);
}

// ===========================================================================
// probe: average line length of the head of the shard -> bytes per tile, so that a tile holds about
// one line per lane of the warp that parses it.  Launched plainly (it zeroes scratch the kernels in front of it
// may have used); the scan kernel is scheduled while it runs and waits for its result.
// ===========================================================================
constexpr int PROBE_THREADS = 1024, PROBE_BYTES = 64 << 10;

__global__ void __launch_bounds__(PROBE_THREADS) probe_kernel(const __grid_constant__ FilterArgs a) {
    cudaTriggerProgrammaticLaunchCompletion();
    __shared__ uint32_t total;
    if (threadIdx.x == 0) total = 0;
    if (threadIdx.x < 16 && threadIdx.x != 4) a.sc.cnt[threadIdx.x] = 0;      // the lists' cursors
    __syncthreads();
    const uint64_t span = a.n < uint64_t(PROBE_BYTES) ? a.n : uint64_t(PROBE_BYTES);
    const uint32_t n16 = uint32_t(span / 16);
    const uint4 *p = reinterpret_cast<const uint4 *>(a.gaf);
    uint32_t cnt = 0;
    for (uint32_t i = threadIdx.x; i < n16; i += PROBE_THREADS) {
        const uint4 v = __ldg(p + i);
        cnt += __popc(eq_bytes(v.x, 0x0A0A0A0Au)) + __popc(eq_bytes(v.y, 0x0A0A0A0Au)) + __popc(eq_bytes(v.z, 0x0A0A0A0Au)) +
               __popc(eq_bytes(v.w, 0x0A0A0A0Au));
    }
    cnt = __reduce_add_sync(0xFFFFFFFFu, cnt);
    if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(&total, cnt);
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t tile_max = a.tile_max;
        uint32_t tile = tile_max;
        if (total) {
            const uint64_t want = uint64_t(n16) * 16ull * a.tile_lines / total;
            tile = uint32_t(want < uint64_t(tile_max) ? want : uint64_t(tile_max)) & ~31u;
        }
        if (const uint32_t forced = (a.flags >> 16)) tile = forced & ~31u;    // SVJG_TUNE_TILE_BYTES
        if (total) {
            // phase A scans 1 KiB a step and stops behind the tile once a line end is found: let a step
            // end about 1.5 lines behind the tile, so that step is rarely followed by one more
            const uint64_t s15 = uint64_t(n16) * 24ull / total;                 // 1.5 lines
            const uint32_t slack = uint32_t(s15 < 512 ? s15 : 512);
            tile = min(tile, tile_max);
            const uint32_t steps = (HEAD + tile + slack) / 1024u;
            if (steps >= 2) tile = (steps * 1024u - HEAD - slack) & ~31u;
        }
        a.sc.cnt[4] = max(uint32_t(TILE_MIN), min(tile, tile_max));
    }
}

__global__ void reset_kernel(uint32_t *counts, uint64_t n, unsigned long long *stats) {
    uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
    uint64_t stride = uint64_t(gridDim.x) * blockDim.x;
    for (uint64_t k = i; k < n; k += stride) counts[k] = 0;
    if (i < 8) stats[i] = (i == 5) ? ~0ull : 0ull;
}

// Launch with programmatic stream serialization: when the work in front of it on the stream is a kernel, this one
// may be scheduled while that kernel still runs (from the point where every block of it has called
// cudaTriggerProgrammaticLaunchCompletion() or exited).  Every thread of a kernel launched so calls
// cudaGridDependencySynchronize() before it reads or writes memory the kernels in front of it use.
template <typename... P, typename... A>
cudaError_t launch_pdl(void (*kernel)(P...), unsigned grid, unsigned block, size_t smem, cudaStream_t st, A &&...args) {
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<A &&>(args)...);
}

// ---- launch configuration, fixed per device the first time a shard is filtered there
struct DevCfg {
    int sms = 0;
    int grid_cap = 0;            // blocks of the scan kernel resident at once (SM count x occupancy)
    int min_blocks = 0;          // the scan kernel's instantiation
    uint32_t tile_max = 0, tile_lines = 0;
    uint32_t smem = 0;           // dynamic shared memory of one block
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;   // around the scan kernel of the last call (svjg_filter_profile)
    bool timed = false;
};
std::mutex g_cfg_mu;
std::map<int, DevCfg> g_cfg;
bool g_profile = false;

// measurement / test knobs (svjg_filter_tune); 0 = default
struct Knobs {
    int tile_bytes = 0, tile_lines = 0, scan_blocks = 0, scan_only = 0, pool_units = 0;
};
Knobs g_knobs;

template <class G>
int configure_scan(DevCfg &c) {
    c.tile_max = G::TILE_MAX;
    c.tile_lines = g_knobs.tile_lines > 0 ? uint32_t(g_knobs.tile_lines) : uint32_t(TILE_LINES);
    c.smem = G::SMEM;
    c.min_blocks = G::MB;
    SVJG_CUDA(cudaFuncSetAttribute(scan_kernel<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(c.smem)));
    int occ = 0;
    SVJG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, scan_kernel<G>, THREADS, c.smem));
    if (occ < 1) return set_error(SVJG_E_CUDA, "scan kernel does not fit on an SM");
    c.grid_cap = c.sms * occ;
    return SVJG_OK;
}

int device_config(DevCfg **out) {
    int dev = 0;
    SVJG_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_cfg_mu);
    auto it = g_cfg.find(dev);
    if (it == g_cfg.end()) {
        DevCfg c;
        SVJG_CUDA(cudaDeviceGetAttribute(&c.sms, cudaDevAttrMultiProcessorCount, dev));
        const int rc = g_knobs.scan_blocks == 8 ? configure_scan<Geo8>(c) : configure_scan<Geo6>(c);
        if (rc) return rc;
        // scratch comes from the device's default memory pool: keep freed blocks cached in the pool
        cudaMemPool_t pool;
        SVJG_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
        uint64_t keep = ~0ull;
        SVJG_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
        SVJG_CUDA(cudaEventCreate(&c.ev0));
        SVJG_CUDA(cudaEventCreate(&c.ev1));
        it = g_cfg.emplace(dev, c).first;
    }
    *out = &it->second;
    return SVJG_OK;
}

}  // namespace

extern "C" int svjg_filter_reset(uint32_t *d_counts, uint32_t num_sv, svjg_filter_stats *d_stats, void *stream) {
    if (!d_counts || !d_stats) return set_error(SVJG_E_ARG, "svjg_filter_reset: NULL argument");
    uint64_t n = uint64_t(num_sv) * 2;
    int blocks = int(std::min<uint64_t>(1184, (n + 255) / 256));
    if (blocks < 1) blocks = 1;
    reset_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(d_counts, n, reinterpret_cast<unsigned long long *>(d_stats));
    SVJG_CUDA(cudaGetLastError());
    return SVJG_OK;
}

extern "C" int svjg_filter_device(const svjg_tables *t, const uint8_t *d_gaf, uint64_t n_bytes, uint64_t base_offset,
                                  int64_t d_over, uint32_t *d_counts, uint32_t *d_hit_sv2, uint32_t *d_hit_off,
                                  uint32_t *d_hit_len, uint64_t hit_cap, svjg_filter_stats *d_stats, void *stream) {
    return svjg::filter_device_abs(t, d_gaf, n_bytes, base_offset, d_over, d_counts, d_hit_sv2, d_hit_off, nullptr, d_hit_len,
                                   hit_cap, d_stats, stream);
}

// Measurement aid: with profiling on, every svjg_filter_device call records CUDA events around its scan
// kernel on the caller's stream; svjg_filter_scan_ms waits for the last such call on the current device
// and gives the kernel's duration.
extern "C" int svjg_filter_tune(int knob, int value) {
    if (value < 0) return set_error(SVJG_E_ARG, "svjg_filter_tune: negative value");
    std::lock_guard<std::mutex> lock(g_cfg_mu);
    switch (knob) {
        case SVJG_TUNE_TILE_BYTES: g_knobs.tile_bytes = value; break;
        case SVJG_TUNE_SCAN_ONLY: g_knobs.scan_only = value; break;
        case SVJG_TUNE_POOL_UNITS: g_knobs.pool_units = value; break;
        case SVJG_TUNE_TILE_LINES:
        case SVJG_TUNE_SCAN_BLOCKS:
            // part of the per-device launch configuration: drop it, the next call configures anew
            if (knob == SVJG_TUNE_TILE_LINES) g_knobs.tile_lines = value;
            else g_knobs.scan_blocks = value;
            for (auto &kv : g_cfg) {
                cudaEventDestroy(kv.second.ev0);
                cudaEventDestroy(kv.second.ev1);
            }
            g_cfg.clear();
            break;
        default: return set_error(SVJG_E_ARG, "svjg_filter_tune: unknown knob");
    }
    return SVJG_OK;
}
extern "C" int svjg_filter_profile(int enable) {
    g_profile = enable != 0;
    return SVJG_OK;
}
extern "C" int svjg_filter_scan_ms(float *ms) {
    if (!ms) return set_error(SVJG_E_ARG, "svjg_filter_scan_ms: NULL argument");
    DevCfg *c = nullptr;
    if (int rc = device_config(&c)) return rc;
    if (!c->timed) return set_error(SVJG_E_ARG, "svjg_filter_scan_ms: no profiled call on this device");
    SVJG_CUDA(cudaEventSynchronize(c->ev1));
    SVJG_CUDA(cudaEventElapsedTime(ms, c->ev0, c->ev1));
    return SVJG_OK;
}

// d_hit_off64 != NULL: absolute 64-bit offsets (base_offset + offset) instead of d_hit_off (svjg_filter_host)
int svjg::filter_device_abs(const svjg_tables *t, const uint8_t *d_gaf, uint64_t n_bytes, uint64_t base_offset, int64_t d_over,
                            uint32_t *d_counts, uint32_t *d_hit_sv2, uint32_t *d_hit_off, uint64_t *d_hit_off64,
                            uint32_t *d_hit_len, uint64_t hit_cap, svjg_filter_stats *d_stats, void *stream, bool inside_buffer) {
    if (!t || t->device < 0) return set_error(SVJG_E_ARG, "svjg_filter_device: tables are not on a device");
    // a shard that starts right behind a line end somewhere inside a larger device buffer: the kernels start at the
    // 16-byte boundary in front of it and see the tail of that line first, which is nobody's line
    uint32_t skip = 0;
    if (inside_buffer) {
        skip = uint32_t(reinterpret_cast<uintptr_t>(d_gaf) & 15);
        if (base_offset < skip) return set_error(SVJG_E_ARG, "svjg_filter_device: shard inside a buffer without the bytes in front of it");
        d_gaf -= skip;
        n_bytes += n_bytes ? skip : 0;
        base_offset -= skip;
    }
    if (!d_counts || !d_stats || (n_bytes && !d_gaf)) return set_error(SVJG_E_ARG, "svjg_filter_device: NULL argument");
    if (hit_cap && (!d_hit_sv2 || (!d_hit_off && !d_hit_off64) || !d_hit_len))
        return set_error(SVJG_E_ARG, "svjg_filter_device: NULL hit buffer");
    if (reinterpret_cast<uintptr_t>(d_gaf) & 15) return set_error(SVJG_E_ARG, "svjg_filter_device: d_gaf must be 16-byte aligned");
    if (n_bytes >= 0xFFFF0000ull) return set_error(SVJG_E_ARG, "svjg_filter_device: shard must be smaller than 4 GiB");
    if (n_bytes == 0) return SVJG_OK;
    cudaStream_t st = (cudaStream_t)stream;
    DevCfg *cfg = nullptr;
    if (int rc = device_config(&cfg)) return rc;
    FilterArgs a;
    a.gaf = d_gaf;
    a.n = n_bytes;
    a.base = base_offset;
    a.d_over = d_over;
    a.tb = t->dev;
    a.counts = d_counts;
    a.hit_sv2 = d_hit_sv2;
    a.hit_off = d_hit_off;
    a.hit_off64 = d_hit_off64;
    a.hit_len = d_hit_len;
    a.hit_cap = hit_cap;
    a.stats = reinterpret_cast<unsigned long long *>(d_stats);
    a.flags = t->filter_flags;
    a.one = 1;
    a.skip = skip;
    a.tile_max = cfg->tile_max;
    a.tile_lines = cfg->tile_lines;
    if (g_knobs.scan_only) a.flags |= FLAG_STOP_AFTER_SCAN;
    if (g_knobs.tile_bytes) a.flags |= uint32_t(std::min(65535, g_knobs.tile_bytes)) << 16;

    // scratch: one stream-ordered allocation, carved into the lists
    Scratch &sc = a.sc;
    sc.cap_exact = uint32_t(n_bytes / 16 + 64);       // a line shorter than 16 bytes cannot hold 12 columns
    sc.cap_pool = uint32_t(std::min<uint64_t>(4u << 20, std::max<uint64_t>(64u << 10, n_bytes / 256)));   // 16-byte units: 1-64 MiB
    if (g_knobs.pool_units) sc.cap_pool = uint32_t(g_knobs.pool_units);
    auto up = [](size_t x) { return (x + 255) & ~size_t(255); };
    const size_t o_cnt = 0, o_ex = up(64), o_slab = o_ex + up(size_t(sc.cap_exact) * 4),
                 o_pool = o_slab + up(size_t(cfg->grid_cap) * WARPS * SLAB_N * sizeof(uint4)),
                 total = o_pool + up(size_t(sc.cap_pool) * sizeof(uint4));
    uint8_t *ws = nullptr;
    SVJG_CUDA(cudaMallocAsync(reinterpret_cast<void **>(&ws), total, st));
    sc.cnt = reinterpret_cast<uint32_t *>(ws + o_cnt);
    sc.exact = reinterpret_cast<uint32_t *>(ws + o_ex);
    sc.slab = reinterpret_cast<uint4 *>(ws + o_slab);
    sc.pool = reinterpret_cast<uint4 *>(ws + o_pool);

    const uint32_t max_tiles = uint32_t((n_bytes + TILE_MIN - 1) / TILE_MIN);
    const int scan_grid = int(std::min<uint32_t>((max_tiles + WARPS - 1) / WARPS, uint32_t(cfg->grid_cap)));
    // with profiling on, the events between the kernels keep them apart: the scan kernel's time is its own
    probe_kernel<<<1, PROBE_THREADS, 0, st>>>(a);
    cudaError_t le = cudaGetLastError();
    if (g_profile) cudaEventRecord(cfg->ev0, st);
    if (le == cudaSuccess)
        le = launch_pdl(cfg->min_blocks == 8 ? scan_kernel<Geo8> : scan_kernel<Geo6>, scan_grid, THREADS, cfg->smem, st, a);
    if (g_profile) cudaEventRecord(cfg->ev1, st), cfg->timed = true;
    if (le == cudaSuccess && !(a.flags & FLAG_STOP_AFTER_SCAN))
        le = launch_pdl(exact_kernel, cfg->sms * 2, FLAT_THREADS, 0, st, a);     // a few lines as a rule: a small grid starts faster
    if (le == cudaSuccess) le = cudaGetLastError();
    cudaError_t fe = cudaFreeAsync(ws, st);
    SVJG_CUDA(le);
    SVJG_CUDA(fe);
    return SVJG_OK;
}
