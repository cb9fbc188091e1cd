// VCF side of the genotype stage on the host: the SV key of every record (predict-genotype.py:118-211),
// the gate inputs of :216 and the output text of :248-271, without a Python-level loop over the records
// (C5: 1 M records).  svjg/genotype.py::parse_vcf / format_vcf are the line-by-line statement of the same
// rules; tests/test_vcf_native.py holds the two against each other on every fixture.
//
// Only spellings whose Python meaning is reproduced exactly are accepted: a file with a non-ASCII
// byte, or a POS/END of more than 18 digits, is answered with SVJG_E_UNSUPPORTED and the caller uses
// the Python statement instead.
#include <cstdio>
#include <algorithm>
#include <cstring>
#include <string>
#include <string_view>
#include <unordered_map>
#include <thread>
#include <vector>

#include "../../include/svjg.h"
#include "svjg_internal.h"

using svjg::set_error;
using sv = std::string_view;

namespace {

const char FORMAT_LINES[] =
    "##FORMAT=<ID=GT,Number=1,Type=String,Description=\"Genotype\">\n"
    "##FORMAT=<ID=DP,Number=1,Type=Float,Description=\"Total number of informative read alignments across all alleles "
    "(after normalization for unbalanced SVs)\">\n"
    "##FORMAT=<ID=AD,Number=2,Type=Float,Description=\"Number of informative read alignments supporting each allele "
    "(after normalization by breakpoint number for unbalanced SVs)\">\n"
    "##FORMAT=<ID=PL,Number=3,Type=Integer,Description=\"Phred-scaled likelihood for each genotype\">\n"
    "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t";      // then the sample names and "\n"

struct Rec {
    uint64_t head_off;   // into text
    uint32_t head_len;
    uint32_t key_len;    // UINT32_MAX: no key
    uint64_t key_off;    // into keys
};
struct Hdr {
    uint32_t before;     // printed in front of this record index
    uint32_t len;        // UINT32_MAX: the FORMAT block + column header
    uint64_t off;
};

inline bool starts_with(sv s, sv p) { return s.size() >= p.size() && memcmp(s.data(), p.data(), p.size()) == 0; }

// s.split(sep)[1] (npos-safe): the text between the first and the second occurrence of sep; false if sep is absent
bool second_piece(sv s, sv sep, sv &out) {
    size_t a = s.find(sep);
    if (a == sv::npos) return false;
    a += sep.size();
    size_t b = s.find(sep, a);
    out = s.substr(a, b == sv::npos ? sv::npos : b - a);
    return true;
}
inline sv upto_semicolon(sv s) {
    size_t p = s.find(';');
    return p == sv::npos ? s : s.substr(0, p);
}
inline sv first_field(sv info) { return upto_semicolon(info); }
inline sv last_field(sv info) {
    size_t p = info.rfind(';');
    return p == sv::npos ? info : info.substr(p + 1);
}

// get_info of predict-genotype.py:77-87; false where the reference raises IndexError
bool info_value(sv info, sv tag /* "END=" */, sv sep_tag /* ";END=" */, sv &out) {
    sv piece;
    if (starts_with(first_field(info), tag)) {
        second_piece(info, tag, piece);
        out = upto_semicolon(piece);
        return true;
    }
    if (!second_piece(info, sep_tag, piece)) return false;
    out = starts_with(last_field(info), tag) ? piece : upto_semicolon(piece);
    return true;
}

inline bool py_space(unsigned char c) { return c == ' ' || (c >= 9 && c <= 13) || (c >= 0x1c && c <= 0x1f); }

// int(str) for ASCII text.  0 ok, 1 ValueError, 2 more than 18 digits
int py_int(sv s, int64_t &out) {
    while (!s.empty() && py_space((unsigned char)s.front())) s.remove_prefix(1);
    while (!s.empty() && py_space((unsigned char)s.back())) s.remove_suffix(1);
    bool neg = false;
    if (!s.empty() && (s.front() == '+' || s.front() == '-')) {
        neg = s.front() == '-';
        s.remove_prefix(1);
    }
    if (s.empty()) return 1;
    int64_t v = 0;
    int digits = 0;
    bool prev_digit = false;
    for (char c : s) {
        if (c >= '0' && c <= '9') {
            if (v || c != '0') {
                if (++digits > 18) return 2;
            }
            v = v * 10 + (c - '0');
            prev_digit = true;
        } else if (c == '_' && prev_digit) {
            prev_digit = false;            // a single underscore between two digits
        } else {
            return 1;
        }
    }
    if (!prev_digit) return 1;             // trailing underscore
    out = neg ? -v : v;
    return 0;
}

}  // namespace

struct svjg_vcf {
    std::string text;                // the file as text mode reads it ("\r\n" and "\r" are "\n")
    std::string keys;
    std::vector<Rec> recs;
    std::vector<uint8_t> type;
    std::vector<Hdr> hdrs;
};

#define SVJG_VCF_FAIL(msg)                                                                             \
    do {                                                                                               \
        delete v;                                                                                      \
        return set_error(SVJG_E_INPUT, std::string("VCF line ") + std::to_string(line_no) + ": " + msg); \
    } while (0)

extern "C" int svjg_vcf_parse(const char *data, size_t len, int translate_cr, svjg_vcf **out) {
    if ((!data && len) || !out) return set_error(SVJG_E_ARG, "svjg_vcf_parse: NULL argument");
    {
        uint64_t acc = 0;
        size_t i = 0;
        for (; i + 8 <= len; i += 8) {
            uint64_t w;
            memcpy(&w, data + i, 8);
            acc |= w;
        }
        for (; i < len; ++i) acc |= uint64_t((unsigned char)data[i]);
        if (acc & 0x8080808080808080ull)
            return set_error(SVJG_E_UNSUPPORTED, "VCF with non-ASCII bytes: left to the Python statement of the rules");
    }
    svjg_vcf *v = new svjg_vcf();
    if (translate_cr && len && memchr(data, '\r', len)) {
        v->text.reserve(len);
        for (size_t i = 0; i < len; ++i) {
            if (data[i] == '\r') {
                v->text.push_back('\n');
                if (i + 1 < len && data[i + 1] == '\n') ++i;
            } else {
                v->text.push_back(data[i]);
            }
        }
    } else {
        v->text.assign(data ? data : "", len);
    }
    const std::string &t = v->text;
    std::unordered_map<std::string, uint32_t> ins_seen;   // running count per POS string, any chromosome (:151-155)
    size_t p = 0, line_no = 0;
    std::string key;
    while (p < t.size()) {
        ++line_no;
        size_t nl = t.find('\n', p);
        const size_t next = nl == std::string::npos ? t.size() : nl + 1;
        const sv line(t.data() + p, next - p);                                  // with its "\n"
        const sv body(t.data() + p, (nl == std::string::npos ? t.size() : nl) - p);   // line.rstrip("\n")
        p = next;
        if (starts_with(line, "##FORMAT")) continue;
        if (starts_with(line, "##")) {
            v->hdrs.push_back({uint32_t(v->recs.size()), uint32_t(line.size()), uint64_t(line.data() - t.data())});
            continue;
        }
        if (starts_with(line, "#C")) {
            v->hdrs.push_back({uint32_t(v->recs.size()), UINT32_MAX, 0});
            continue;
        }
        // columns 0..7 and where the 8th ends
        sv col[8];
        size_t a = 0;
        int nc = 0;
        size_t end8 = sv::npos;      // offset of the tab after column 7, npos if the line has exactly 8 columns
        while (nc < 8) {
            size_t tab = body.find('\t', a);
            if (tab == sv::npos) {
                col[nc++] = body.substr(a);
                a = sv::npos;
                break;
            }
            col[nc++] = body.substr(a, tab - a);
            a = tab + 1;
            if (nc == 8) end8 = tab;
        }
        if (nc < 8) SVJG_VCF_FAIL("fewer than 8 columns");
        const sv chrom = col[0], pos = col[1], alt = col[4], info = col[7];
        sv svtype;
        if (info.find("SVTYPE") != sv::npos) {
            sv piece;
            if (!second_piece(info, "SVTYPE=", piece)) SVJG_VCF_FAIL("SVTYPE without a value");
            svtype = starts_with(last_field(info), "SVTYPE=") ? piece : upto_semicolon(piece);
        }
        const bool is_del = svtype == "DEL", is_inv = svtype == "INV", is_ins = svtype == "INS", is_bnd = svtype == "BND";
        bool has_key = false;
        bool is_short = false;          // |length| < 50
        key.clear();
        if (!is_bnd && !is_ins) {
            sv end;
            if (!info_value(info, "END=", ";END=", end)) SVJG_VCF_FAIL("INFO has no END=");
            if (is_del || is_inv) {
                int64_t e = 0, s = 0;
                const int r1 = py_int(end, e), r2 = py_int(pos, s);
                if (r1 == 1) SVJG_VCF_FAIL("non-integer POS/END");      // int(end) is evaluated first
                if (r1 == 2) {
                    delete v;
                    return set_error(SVJG_E_UNSUPPORTED, "POS/END of more than 18 digits: left to the Python statement of the rules");
                }
                if (r2 == 1) SVJG_VCF_FAIL("non-integer POS/END");
                if (r2 == 2) {
                    delete v;
                    return set_error(SVJG_E_UNSUPPORTED, "POS/END of more than 18 digits: left to the Python statement of the rules");
                }
                const int64_t d = e - s;
                is_short = d > -50 && d < 50;
                key.append(chrom).append(":").append(svtype).append("-").append(pos).append("-").append(end);
                has_key = true;
            }
        } else if (is_ins) {
            const uint32_t k = ++ins_seen[std::string(pos)];
            key.append(chrom).append(":INS-").append(pos).append("-").append(std::to_string(k));
            has_key = true;
            is_short = alt.size() < 50;                                   // len(ALT), ASCII
        } else {
            key = "wrong_format";
            has_key = true;
            for (char br : {'[', ']'}) {
                if (alt.find(br) == sv::npos) continue;
                sv piece[2];
                int np = 0;
                size_t b = 0;
                while (b <= alt.size() && np < 2) {                       // the first two non-empty pieces of alt.split(br)
                    size_t e = alt.find(br, b);
                    if (e == sv::npos) e = alt.size();
                    if (e > b) piece[np++] = alt.substr(b, e - b);
                    b = e + 1;
                }
                if (np < 2) SVJG_VCF_FAIL("malformed BND ALT");
                key.clear();
                key.append(chrom).append(":BND-");
                if (piece[1].find(':') != sv::npos)
                    key.append(pos).append(1, br).append(piece[1]).append(1, br);
                else
                    key.append(1, br).append(piece[0]).append(1, br).append(pos);
                break;
            }
        }
        uint8_t code = is_del ? 0 : is_ins ? 1 : is_inv ? 2 : is_bnd ? 3 : 255;
        if (code != 255 && is_short) code |= 0x80;
        Rec r{};
        r.head_off = uint64_t(body.data() - t.data());
        r.head_len = uint32_t(end8 == sv::npos ? body.size() : end8);
        if (has_key) {
            r.key_off = v->keys.size();
            r.key_len = uint32_t(key.size());
            v->keys.append(key);
        } else {
            r.key_len = UINT32_MAX;
        }
        if (v->recs.size() >= 0xFFFFFFF0u) SVJG_VCF_FAIL("too many records");
        v->recs.push_back(r);
        v->type.push_back(code);
    }
    *out = v;
    return SVJG_OK;
}

extern "C" void svjg_vcf_free(svjg_vcf *v) { delete v; }
extern "C" uint32_t svjg_vcf_num_records(const svjg_vcf *v) { return v ? uint32_t(v->recs.size()) : 0; }
extern "C" const uint8_t *svjg_vcf_svtype(const svjg_vcf *v) { return v ? v->type.data() : nullptr; }
extern "C" const char *svjg_vcf_key(const svjg_vcf *v, uint32_t i, uint32_t *len) {
    if (!v || i >= v->recs.size() || v->recs[i].key_len == UINT32_MAX) return nullptr;
    if (len) *len = v->recs[i].key_len;
    return v->keys.data() + v->recs[i].key_off;
}

extern "C" int svjg_vcf_index_tables(const svjg_vcf *v, const svjg_tables *t, uint32_t *sv_index) {
    if (!v || !t || (!sv_index && !v->recs.empty())) return set_error(SVJG_E_ARG, "svjg_vcf_index_tables: NULL argument");
    for (size_t i = 0; i < v->recs.size(); ++i) {
        const Rec &r = v->recs[i];
        sv_index[i] = r.key_len == UINT32_MAX ? UINT32_MAX : svjg_tables_find_sv(t, v->keys.data() + r.key_off, r.key_len);
    }
    return SVJG_OK;
}

extern "C" int svjg_vcf_index_counts(const svjg_vcf *v, const svjg_aln_counts *c, uint32_t *sv_index, uint8_t *svtype) {
    if (!v || !c || ((!sv_index || !svtype) && !v->recs.empty())) return set_error(SVJG_E_ARG, "svjg_vcf_index_counts: NULL argument");
    const uint32_t *counts = svjg_aln_counts_data(c);
    for (size_t i = 0; i < v->recs.size(); ++i) {
        const Rec &r = v->recs[i];
        uint8_t ty = v->type[i];
        sv_index[i] = UINT32_MAX;
        svtype[i] = ty;
        if (r.key_len == UINT32_MAX) continue;
        const uint32_t j = svjg_aln_counts_find(c, v->keys.data() + r.key_off, r.key_len);
        if (j == UINT32_MAX) continue;
        const bool gated = ty != 255 && (ty & 0x3F) <= 3 && !(ty & 0x80);
        if (gated && counts[size_t(j) * 2] == UINT32_MAX)
            return set_error(SVJG_E_INPUT, "informative_aln entry of '" + std::string(v->keys.data() + r.key_off, r.key_len) +
                                               "' is not a pair of lists (the reference raises here)");
        sv_index[i] = j;
        if (ty != 255) svtype[i] = ty | 0x40;
    }
    return SVJG_OK;
}

namespace {
inline char *put_u64(char *o, uint64_t x) {
    char b[24];
    int n = 0;
    do {
        b[n++] = char('0' + x % 10);
        x /= 10;
    } while (x);
    while (n) *o++ = b[--n];
    return o;
}
inline char *put_i64(char *o, int64_t x) {
    if (x < 0) {
        *o++ = '-';
        return put_u64(o, uint64_t(0) - uint64_t(x));
    }
    return put_u64(o, uint64_t(x));
}
// str() of a count held in half units: int when the allele was not normalised, else one decimal
inline char *put_half(char *o, uint64_t twice, bool halved) {
    o = put_u64(o, twice >> 1);
    if (halved) {
        *o++ = '.';
        *o++ = (twice & 1) ? '5' : '0';
    }
    return o;
}
inline char *put_mem(char *o, const char *p, size_t n) {
    memcpy(o, p, n);
    return o + n;
}

// The population INFO tags of a cohort VCF, in the order they are written (bit k of the mask is entry k), with the
// header lines bcftools +fill-tags writes for them, so that filter expressions written for those read the same.
struct InfoTag {
    sv id;
    bool per_alt;       // Number=A
    const char *hdr;
};
const InfoTag INFO_TAGS[] = {
    {"NS", false, "##INFO=<ID=NS,Number=1,Type=Integer,Description=\"Number of samples with data\">\n"},
    {"AN", false, "##INFO=<ID=AN,Number=1,Type=Integer,Description=\"Total number of alleles in called genotypes\">\n"},
    {"AC", true, "##INFO=<ID=AC,Number=A,Type=Integer,Description=\"Allele count in genotypes\">\n"},
    {"AF", true, "##INFO=<ID=AF,Number=A,Type=Float,Description=\"Allele frequency\">\n"},
    {"AC_Het", true, "##INFO=<ID=AC_Het,Number=A,Type=Integer,Description=\"Allele counts in heterozygous genotypes\">\n"},
    {"AC_Hom", true, "##INFO=<ID=AC_Hom,Number=A,Type=Integer,Description=\"Allele counts in homozygous genotypes\">\n"},
    {"F_MISSING", false, "##INFO=<ID=F_MISSING,Number=1,Type=Float,Description=\"Fraction of missing genotypes\">\n"},
    {"HWE", true, "##INFO=<ID=HWE,Number=A,Type=Float,Description=\"HWE test (PMID:15789306); 1=good, 0=bad\">\n"},
    {"ExcHet", true, "##INFO=<ID=ExcHet,Number=A,Type=Float,Description=\"Test excess heterozygosity; 1=good, 0=bad\">\n"},
};
constexpr uint32_t N_INFO_TAGS = sizeof INFO_TAGS / sizeof INFO_TAGS[0];

bool selected_tag(uint32_t tags, sv key) {
    for (uint32_t t = 0; t < N_INFO_TAGS; ++t)
        if ((tags >> t & 1) && key == INFO_TAGS[t].id) return true;
    return false;
}

// "##INFO=<ID=X," or "##INFO=<ID=X>" for a selected X
bool info_header_of(uint32_t tags, sv line) {
    if (!starts_with(line, "##INFO=<ID=")) return false;
    const sv rest = line.substr(11);
    const size_t e = rest.find_first_of(",>");
    return e != sv::npos && selected_tag(tags, rest.substr(0, e));
}

// The value text of tag t for counts g = (r0, h, r2, m) of S cells; "." where it has none
size_t tag_value(char *o, uint32_t t, const uint32_t *g, uint64_t S, double hwe, double exchet, bool multi_alt) {
    if (INFO_TAGS[t].per_alt && multi_alt) {
        *o = '.';
        return 1;
    }
    const uint64_t r0 = g[0], h = g[1], r2 = g[2], m = g[3], ns = r0 + h + r2;
    auto num = [&](uint64_t x) { return size_t(put_u64(o, x) - o); };
    auto flt = [&](bool have, double x) -> size_t {
        if (!have) {
            *o = '.';
            return 1;
        }
        return size_t(snprintf(o, 32, "%.6g", x));
    };
    switch (1u << t) {
        case SVJG_TAG_NS: return num(ns);
        case SVJG_TAG_AN: return num(2 * ns);
        case SVJG_TAG_AC: return num(h + 2 * r2);
        case SVJG_TAG_AF: return flt(ns != 0, double(h + 2 * r2) / double(2 * ns));
        case SVJG_TAG_AC_HET: return num(h);
        case SVJG_TAG_AC_HOM: return num(2 * r2);
        case SVJG_TAG_F_MISSING: return flt(true, double(m) / double(S));
        case SVJG_TAG_HWE: return flt(ns != 0, hwe);
        default: return flt(ns != 0, exchet);
    }
}
}  // namespace

// Records [lo, hi) with one column per sample; the arrays hold those records' cells, [hi - lo][S].
extern "C" int svjg_vcf_format_cohort_tags(const svjg_vcf *v, uint32_t lo, uint32_t hi, uint32_t n_samples, const char *names,
                                           uint64_t names_len, const uint8_t *gt, const uint8_t *flags, const uint32_t *ad2,
                                           const int64_t *pl, uint32_t tags, const uint32_t *gcount, const double *hwe,
                                           const double *exchet, char **out, uint64_t *out_len, uint64_t *n_genotyped) {
    if (!v || !out || !out_len || !names || !n_genotyped) return set_error(SVJG_E_ARG, "svjg_vcf_format: NULL argument");
    const size_t n_all = v->recs.size();
    if (lo > hi || hi > n_all || n_samples == 0) return set_error(SVJG_E_ARG, "svjg_vcf_format: bad record range or sample count");
    const size_t S = n_samples, n = size_t(hi - lo), n_cells = n * S;
    if (n && (!gt || !flags || !ad2 || !pl)) return set_error(SVJG_E_ARG, "svjg_vcf_format: NULL argument");
    if (tags >> N_INFO_TAGS) return set_error(SVJG_E_ARG, "svjg_vcf_format: unknown INFO tag bit");
    // every tag needs the counts (HWE and ExcHet are "." when NS = 0)
    if (n && tags && (!gcount || ((tags & SVJG_TAG_HWE) && !hwe) || ((tags & SVJG_TAG_EXCHET) && !exchet)))
        return set_error(SVJG_E_ARG, "svjg_vcf_format: NULL site statistics");
    if (tags) {
        for (size_t j = 0; j < n; ++j)
            if (uint64_t(gcount[4 * j]) + gcount[4 * j + 1] + gcount[4 * j + 2] + gcount[4 * j + 3] != S)
                return set_error(SVJG_E_ARG, "svjg_vcf_format: genotype counts do not add up to the sample count");
    }
    for (size_t k = 0; k < n_cells; ++k)
        if ((flags[k] & SVJG_GT_GENOTYPED) && gt[k] > 3) return set_error(SVJG_E_ARG, "svjg_vcf_format: gt code out of range");
    static const char *GT_TEXT[4] = {"0/0", "0/1", "1/1", "./."};
    const char *text = v->text.data();
    std::string info_hdr;                  // the ##INFO lines of the selected tags, in front of the ##FORMAT lines
    for (uint32_t t = 0; t < N_INFO_TAGS; ++t)
        if (tags >> t & 1) info_hdr += INFO_TAGS[t].hdr;
    // the header lines of the range: those in front of its records and, for the last range, the ones behind them
    size_t h_lo = 0;
    while (h_lo < v->hdrs.size() && v->hdrs[h_lo].before < lo) ++h_lo;
    size_t h_hi = h_lo;
    while (h_hi < v->hdrs.size() && (hi == n_all || v->hdrs[h_hi].before < hi)) ++h_hi;
    const size_t col_hdr = info_hdr.size() + sizeof FORMAT_LINES - 1 + names_len + 1;
    auto dropped = [&](const Hdr &h) { return tags && info_header_of(tags, sv(text + h.off, h.len)); };
    auto hdr_len = [&](const Hdr &h) -> uint64_t { return h.len == UINT32_MAX ? col_hdr : dropped(h) ? 0 : h.len; };
    auto put_hdr = [&](char *o, const Hdr &h) {
        if (h.len != UINT32_MAX) return dropped(h) ? o : put_mem(o, text + h.off, h.len);
        o = put_mem(o, info_hdr.data(), info_hdr.size());
        o = put_mem(o, FORMAT_LINES, sizeof FORMAT_LINES - 1);
        o = put_mem(o, names, names_len);
        *o++ = '\n';
        return o;
    };
    // columns 1-8 of record lo + j: as the catalogue has them, or with the INFO column rewritten for the tags.
    // o == nullptr: the length only
    auto put_head = [&](char *o, size_t j) -> uint64_t {
        const Rec &r = v->recs[lo + j];
        const sv head(text + r.head_off, r.head_len);
        uint64_t len = 0;
        auto put = [&](const char *p, size_t k) {
            if (o) memcpy(o + len, p, k);
            len += k;
        };
        if (!tags) {
            put(head.data(), head.size());
            return len;
        }
        const size_t t7 = head.rfind('\t');            // the head has 8 columns: INFO is the last
        put(head.data(), t7 + 1);
        const sv info = head.substr(t7 + 1);
        bool first = true;
        if (!info.empty() && info != ".") {
            for (size_t a = 0;;) {
                size_t b = info.find(';', a);
                if (b == sv::npos) b = info.size();
                const sv item = info.substr(a, b - a);
                if (!selected_tag(tags, item.substr(0, item.find('=')))) {
                    if (!first) put(";", 1);
                    put(item.data(), item.size());
                    first = false;
                }
                if (b == info.size()) break;
                a = b + 1;
            }
        }
        size_t a = 0;
        for (int c = 0; c < 4; ++c) a = head.find('\t', a) + 1;   // ALT: column 5
        const bool multi_alt = head.substr(a, head.find('\t', a) - a).find(',') != sv::npos;
        char val[40];
        for (uint32_t t = 0; t < N_INFO_TAGS; ++t) {
            if (!(tags >> t & 1)) continue;
            if (!first) put(";", 1);
            first = false;
            put(INFO_TAGS[t].id.data(), INFO_TAGS[t].id.size());
            put("=", 1);
            put(val, tag_value(val, t, gcount + 4 * j, S, hwe ? hwe[j] : 0.0, exchet ? exchet[j] : 0.0, multi_alt));
        }
        return len;
    };
    // the text of cell k (at most 136 bytes)
    auto put_sample = [&](char *o, size_t k) {
        const uint8_t f = flags[k];
        if (f & SVJG_GT_GENOTYPED) {
            const uint64_t t1 = ad2[2 * k], t2 = ad2[2 * k + 1];
            const bool h0 = f & SVJG_GT_HALVED_0, h1 = f & SVJG_GT_HALVED_1;
            o = put_mem(o, GT_TEXT[gt[k]], 3);
            *o++ = ':';
            o = put_half(o, t1 + t2, h0 || h1);
            *o++ = ':';
            o = put_half(o, t1, h0);
            *o++ = ',';
            o = put_half(o, t2, h1);
            *o++ = ':';
            o = put_i64(o, pl[3 * k]);
            *o++ = ',';
            o = put_i64(o, pl[3 * k + 1]);
            *o++ = ',';
            o = put_i64(o, pl[3 * k + 2]);
        } else {
            o = put_mem(o, "./.:0:0,0:.,.,.", 15);
        }
        return o;
    };
    // what follows the head of record lo + j: the FORMAT column and one column per sample
    auto put_columns = [&](char *o, size_t j) {
        o = put_mem(o, "\tGT:DP:AD:PL", 12);
        for (size_t s = 0; s < S; ++s) {
            *o++ = '\t';
            o = put_sample(o, j * S + s);
        }
        *o++ = '\n';
        return o;
    };
    // where every record starts: its head is copied as it is, the cells are rendered once to learn their
    // length (cheap next to the copies); then the records are filled in by several threads
    std::vector<uint64_t> at(n + 1, 0), genotyped(S, 0);
    {
        char tmp[160];
        size_t h = h_lo;
        uint64_t pos = 0;
        for (size_t j = 0; j < n; ++j) {
            while (h < h_hi && v->hdrs[h].before <= lo + j) pos += hdr_len(v->hdrs[h++]);
            at[j] = pos;
            pos += put_head(nullptr, j) + 13 + S;
            for (size_t s = 0; s < S; ++s) {
                const size_t k = j * S + s;
                genotyped[s] += (flags[k] & SVJG_GT_GENOTYPED) != 0;
                pos += uint64_t(put_sample(tmp, k) - tmp);
            }
        }
        at[n] = pos;
    }
    uint64_t tail = 0;
    {
        size_t h = h_lo;
        while (h < h_hi && (n != 0 && v->hdrs[h].before <= hi - 1)) ++h;
        for (; h < h_hi; ++h) tail += hdr_len(v->hdrs[h]);
    }
    char *buf = (char *)malloc(at[n] + tail + 1);
    if (!buf) return set_error(SVJG_E_NOMEM, "svjg_vcf_format: out of memory");
    auto fill = [&](size_t a, size_t b) {
        size_t h = h_lo;
        while (h < h_hi && v->hdrs[h].before < lo + a) ++h;               // header lines in front of record a: not ours
        // (those with before == lo + a sit right in front of it: ours, they end where it starts)
        for (size_t j = a; j < b; ++j) {
            uint64_t back = 0;
            size_t h2 = h;
            while (h2 < h_hi && v->hdrs[h2].before <= lo + j) back += hdr_len(v->hdrs[h2++]);
            char *o = buf + at[j] - back;
            while (h < h2) o = put_hdr(o, v->hdrs[h++]);
            o += put_head(o, j);
            put_columns(o, j);
        }
    };
    const uint64_t body = at[n];
    unsigned n_thr = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    if (body < (4u << 20) || n < 64) n_thr = 1;
    if (n_thr == 1) {
        fill(0, n);
    } else {
        // ranges of about equal bytes
        std::vector<size_t> cutv(n_thr + 1, 0);
        for (unsigned p = 1; p < n_thr; ++p)
            cutv[p] = size_t(std::lower_bound(at.begin(), at.begin() + n, body * p / n_thr) - at.begin());
        cutv[n_thr] = n;
        for (unsigned p = 1; p <= n_thr; ++p) cutv[p] = std::max(cutv[p], cutv[p - 1]);
        std::vector<std::thread> pool;
        for (unsigned p = 1; p < n_thr; ++p) pool.emplace_back(fill, cutv[p], cutv[p + 1]);
        fill(cutv[0], cutv[1]);
        for (auto &th : pool) th.join();
    }
    // header lines behind the last record of the range
    char *o = buf + at[n];
    {
        size_t h = h_lo;
        while (h < h_hi && (n != 0 && v->hdrs[h].before <= hi - 1)) ++h;
        while (h < h_hi) o = put_hdr(o, v->hdrs[h++]);
    }
    *out = buf;
    *out_len = uint64_t(o - buf);
    for (size_t s = 0; s < S; ++s) n_genotyped[s] += genotyped[s];
    return SVJG_OK;
}

extern "C" int svjg_vcf_format_cohort(const svjg_vcf *v, uint32_t lo, uint32_t hi, uint32_t n_samples, const char *names,
                                      uint64_t names_len, const uint8_t *gt, const uint8_t *flags, const uint32_t *ad2,
                                      const int64_t *pl, char **out, uint64_t *out_len, uint64_t *n_genotyped) {
    return svjg_vcf_format_cohort_tags(v, lo, hi, n_samples, names, names_len, gt, flags, ad2, pl, 0, nullptr, nullptr, nullptr,
                                       out, out_len, n_genotyped);
}

extern "C" int svjg_vcf_format(const svjg_vcf *v, const uint8_t *gt, const uint8_t *flags, const uint32_t *ad2,
                               const int64_t *pl, char **out, uint64_t *out_len, uint64_t *n_genotyped) {
    if (!v) return set_error(SVJG_E_ARG, "svjg_vcf_format: NULL argument");
    uint64_t genotyped = 0;
    const int rc = svjg_vcf_format_cohort(v, 0, uint32_t(v->recs.size()), 1, "SAMPLE", 6, gt, flags, ad2, pl, out, out_len,
                                          &genotyped);
    if (rc == SVJG_OK && n_genotyped) *n_genotyped = genotyped;
    return rc;
}

extern "C" void svjg_buffer_free(char *p) { free(p); }
